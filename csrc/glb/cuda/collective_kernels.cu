// Data-movement collectives over NVLink peer memory (sm_100a): broadcast,
// allgather(v), alltoall(v), reduce_scatter, reduce, gather(v), scatter. All are
// single kernels bracketed by device-side flag barriers; payload moves with
// 128-bit peer loads/stores (or multimem.st through the NVSwitch where a multicast
// alias exists). None of these has a CUDA variant in the reference (SURVEY §0.6).
#include "glb/cuda/bulk_copy.cuh"
#include "glb/cuda/device_common.cuh"
#include "glb/cuda/dispatch.cuh"
#include "glb/cuda/kernels.h"

namespace glb {
namespace cuda {

namespace {

template <typename W>
__device__ __forceinline__ void gridCopyWords(char* dst, const char* src, size_t bytes, size_t tid, size_t nthreads) {
  const size_t n = bytes / sizeof(W);
  constexpr int U = 4;
  for (size_t i0 = tid; i0 < n; i0 += nthreads * U) {
    W w[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t i = i0 + u * nthreads;
      if (i < n) w[u] = reinterpret_cast<const W*>(src)[i];
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t i = i0 + u * nthreads;
      if (i < n) reinterpret_cast<W*>(dst)[i] = w[u];
    }
  }
  for (size_t i = n * sizeof(W) + tid; i < bytes; i += nthreads) dst[i] = src[i];
}

// 16 bytes from a source that is only W-byte aligned (W = 8 or 4), as one pack.
template <typename W>
__device__ __forceinline__ Pack16 ldPackWords(const char* src) {
  Pack16 p;
  W* w = reinterpret_cast<W*>(&p);
#pragma unroll
  for (int i = 0; i < static_cast<int>(16 / sizeof(W)); i++) w[i] = reinterpret_cast<const W*>(src)[i];
  return p;
}

template <typename W>
__device__ __forceinline__ void gridCopyBody(char* dst, const char* src, size_t nvec, size_t tid, size_t nthreads) {
  constexpr int U = 4;
  for (size_t v0 = tid; v0 < nvec; v0 += nthreads * U) {
    Pack16 p[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t v = v0 + u * nthreads;
      if (v < nvec) {
        if constexpr (sizeof(W) == 16) {
          p[u] = ld128_stream(src + v * 16);
        } else {
          p[u] = ldPackWords<W>(src + v * 16);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t v = v0 + u * nthreads;
      if (v < nvec) st128_stream(dst + v * 16, p[u]);
    }
  }
}

// Body copy for a source that is 4-byte (not 8-byte) congruent with the 16-byte aligned
// destination: instead of four 4-byte loads per pack, load the two ALIGNED packs that straddle
// it and pick the words (the second load of one pack is the first load of the next and hits L1/L2).
// The first and last pack use word loads so that no byte outside [src, src + 16 * nvec) is read.
__device__ __forceinline__ void gridCopyBodyShifted(char* dst, const char* src, size_t nvec, size_t tid, size_t nthreads) {
  const int shift = static_cast<int>((reinterpret_cast<uintptr_t>(src) % 16) / 4);  // 1..3 words
  const char* base = src - shift * 4;                                                // 16-byte aligned
  if (tid == 0 && nvec > 0) st128_stream(dst, ldPackWords<unsigned int>(src));
  if (tid == 1 % nthreads && nvec > 1) st128_stream(dst + (nvec - 1) * 16, ldPackWords<unsigned int>(src + (nvec - 1) * 16));
  constexpr int U = 4;
  for (size_t v0 = 1 + tid; v0 + 1 < nvec; v0 += nthreads * U) {
    Pack16 lo[U], hi[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t v = v0 + u * nthreads;
      if (v + 1 < nvec) {
        lo[u] = ld128(base + v * 16);
        hi[u] = ld128(base + v * 16 + 16);
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t v = v0 + u * nthreads;
      if (v + 1 < nvec) {
        Pack16 o;
        if (shift == 1) {
          o.w[0] = lo[u].w[1]; o.w[1] = lo[u].w[2]; o.w[2] = lo[u].w[3]; o.w[3] = hi[u].w[0];
        } else if (shift == 2) {
          o.w[0] = lo[u].w[2]; o.w[1] = lo[u].w[3]; o.w[2] = hi[u].w[0]; o.w[3] = hi[u].w[1];
        } else {
          o.w[0] = lo[u].w[3]; o.w[1] = hi[u].w[0]; o.w[2] = hi[u].w[1]; o.w[3] = hi[u].w[2];
        }
        st128_stream(dst + v * 16, o);
      }
    }
  }
}

// Copy `bytes` from src to dst with the whole grid. The DESTINATION side (usually a peer,
// i.e. NVLink stores) always moves in 128-bit stores: a byte-wise head brings dst to a
// 16-byte boundary, the body loads with the widest access the (local) source allows at
// that point (16 / 8 / 4 bytes) and a byte-wise tail finishes. Only sources that are
// not even 4-byte congruent with the destination fall back to narrow word copies.
__device__ __forceinline__ void gridCopy(char* dst, const char* src, size_t bytes, bool /*vecHint*/, size_t tid,
                                         size_t nthreads) {
  const size_t mis = reinterpret_cast<uintptr_t>(dst) % 16;
  size_t head = mis ? 16 - mis : 0;
  if (head > bytes) head = bytes;
  const uintptr_t srcBody = reinterpret_cast<uintptr_t>(src + head) % 16;
  if (srcBody % 4 != 0) {
    const uintptr_t both = reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src);
    if (both % 2 == 0) {
      gridCopyWords<unsigned short>(dst, src, bytes, tid, nthreads);
    } else {
      for (size_t i = tid; i < bytes; i += nthreads) dst[i] = src[i];
    }
    return;
  }
  for (size_t i = tid; i < head; i += nthreads) dst[i] = src[i];
  const size_t nvec = (bytes - head) / 16;
  if (srcBody == 0) {
    gridCopyBody<Pack16>(dst + head, src + head, nvec, tid, nthreads);
  } else if (srcBody % 8 == 0) {
    gridCopyBody<unsigned long long>(dst + head, src + head, nvec, tid, nthreads);
  } else {
    gridCopyBodyShifted(dst + head, src + head, nvec, tid, nthreads);
  }
  for (size_t i = head + nvec * 16 + tid; i < bytes; i += nthreads) dst[i] = src[i];
}

}  // namespace

// ---- broadcast -----------------------------------------------------------------------
// mode 0: root pushes the whole buffer to every peer (latency regime).
// mode 1: scatter + allgather: root pushes slice i to rank i, then every rank
//         pushes its slice to the others; per-GPU egress ~S instead of (P-1)·S.
// mode 2: NVLS: root issues multimem.st, the switch replicates.
// mode 3: relay, chunk-pipelined: the buffer is cut into chunks of (P-1) slices; the root
//         sends slice j of a chunk to relay j ONLY and raises a per-chunk flag; relay j
//         forwards its slice to the other P-2 ranks while the root is already sending the
//         next chunk. Root egress = S, every other GPU's ingress = S and egress
//         S(P-2)/(P-1): all links run at once, nothing is sent twice over the same port
//         (measured on 8 x B200: a single multimem.st source tops out at ~390 GB/s, NCCL's
//         ring broadcast at ~650).
__global__ void __launch_bounds__(kThreads, 2)
broadcastKernel(CommArgs a, PeerPtrs bufs, char* mc, size_t bytes, int root, int mode, bool vec, int tile) {
  const uint32_t e = loadEpoch(a);
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const int P = a.nranks;
  uint32_t used = mode == 1 ? 3 : 2;
  const size_t relayChunk = static_cast<size_t>(P - 1) * gridDim.x * static_cast<size_t>(tile);  // 16-byte units
  const uint32_t nchunks = mode == 3 ? static_cast<uint32_t>((bytes / 16 + relayChunk - 1) / relayChunk) : 0u;
  if (mode == 3) used = nchunks + 2;  // one flag value per chunk between the two barriers
  if (!blockBarrier<false>(a, e + 1)) {  // every destination may now be overwritten
    retire(a, used, 0);
    return;
  }
  if (mode == 0) {
    if (a.rank == root) {
      const char* src = static_cast<const char*>(bufs.p[root]);
      const size_t nvec = vec ? bytes / 16 : 0;
      constexpr int U = 4;
      for (size_t v0 = tid; v0 < nvec; v0 += nthreads * U) {
        Pack16 p[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
          const size_t v = v0 + u * nthreads;
          if (v < nvec) p[u] = ld128_stream(src + v * 16);
        }
        for (int i = 1; i < P; i++) {
          char* dst = static_cast<char*>(bufs.p[(root + i) % P]);
#pragma unroll
          for (int u = 0; u < U; u++) {
            const size_t v = v0 + u * nthreads;
            if (v < nvec) st128_stream(dst + v * 16, p[u]);
          }
        }
      }
      for (size_t i = nvec * 16 + tid; i < bytes; i += nthreads) {
        const char c = src[i];
        for (int r = 1; r < P; r++) static_cast<char*>(bufs.p[(root + r) % P])[i] = c;
      }
    }
  } else if (mode == 2) {
    if (a.rank == root) {
      const char* src = static_cast<const char*>(bufs.p[root]);
      const size_t nvec = bytes / 16;
      constexpr int U = 4;
      for (size_t v0 = tid; v0 < nvec; v0 += nthreads * U) {
        Pack16 p[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
          const size_t v = v0 + u * nthreads;
          if (v < nvec) p[u] = ld128_stream(src + v * 16);
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
          const size_t v = v0 + u * nthreads;
          if (v < nvec) multimemSt128(mc + v * 16, p[u]);
        }
      }
      for (size_t i = nvec * 16 + tid; i < bytes; i += nthreads) {
        const char c = src[i];
        for (int r = 1; r < P; r++) static_cast<char*>(bufs.p[(root + r) % P])[i] = c;
      }
    }
  } else if (mode == 3) {
    const size_t units = bytes / 16;
    const int R = P - 1;
    constexpr int U = 4;
    if (a.rank == root) {
      const char* src = static_cast<const char*>(bufs.p[root]);
      for (uint32_t c = 0; c < nchunks; c++) {
        for (int j = 0; j < R; j++) {
          const size_t lo = ((static_cast<size_t>(c) * R + j) * gridDim.x + blockIdx.x) * tile;
          if (lo >= units) continue;
          const size_t n = units - lo < static_cast<size_t>(tile) ? units - lo : static_cast<size_t>(tile);
          char* dst = static_cast<char*>(bufs.p[(root + 1 + j) % P]) + lo * 16;
          const char* s = src + lo * 16;
          for (size_t v0 = threadIdx.x; v0 < n; v0 += static_cast<size_t>(blockDim.x) * U) {
            Pack16 p[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
              const size_t v = v0 + static_cast<size_t>(u) * blockDim.x;
              if (v < n) p[u] = ld128_stream(s + v * 16);
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
              const size_t v = v0 + static_cast<size_t>(u) * blockDim.x;
              if (v < n) st128_stream(dst + v * 16, p[u]);
            }
          }
        }
        __syncthreads();
        if (static_cast<int>(threadIdx.x) < R) {
          st_release_sys(&a.sig[(root + 1 + threadIdx.x) % P]->flag[blockIdx.x][root], e + 2 + c);
        }
      }
      for (size_t i = units * 16 + tid; i < bytes; i += nthreads) {
        const char ch = src[i];
        for (int r = 1; r < P; r++) static_cast<char*>(bufs.p[(root + r) % P])[i] = ch;
      }
    } else {
      const int j = (a.rank - root - 1 + P) % P;
      const char* src = static_cast<const char*>(bufs.p[a.rank]);
      for (uint32_t c = 0; c < nchunks; c++) {
        int ok = 1;
        if (threadIdx.x == 0) ok = waitFlag(a, &a.self->flag[blockIdx.x][root], e + 2 + c, root) ? 1 : 0;
        if (!__syncthreads_and(ok)) break;
        const size_t lo = ((static_cast<size_t>(c) * R + j) * gridDim.x + blockIdx.x) * tile;
        if (lo >= units) continue;
        const size_t n = units - lo < static_cast<size_t>(tile) ? units - lo : static_cast<size_t>(tile);
        const char* s = src + lo * 16;
        for (size_t v0 = threadIdx.x; v0 < n; v0 += static_cast<size_t>(blockDim.x) * U) {
          Pack16 p[U];
#pragma unroll
          for (int u = 0; u < U; u++) {
            const size_t v = v0 + static_cast<size_t>(u) * blockDim.x;
            if (v < n) p[u] = ld128_stream(s + v * 16);
          }
          for (int i = 1; i < P; i++) {
            const int d = (a.rank + i) % P;
            if (d == root) continue;
            char* dst = static_cast<char*>(bufs.p[d]) + lo * 16;
#pragma unroll
            for (int u = 0; u < U; u++) {
              const size_t v = v0 + static_cast<size_t>(u) * blockDim.x;
              if (v < n) st128_stream(dst + v * 16, p[u]);
            }
          }
        }
      }
    }
  } else {
    // Slices are 16-byte granular so every phase stays vectorised.
    const size_t units = bytes / 16;
    if (a.rank == root) {
      for (int i = 1; i < P; i++) {
        const int dst = (root + i) % P;
        size_t b, en;
        shareOf(units, P, dst, b, en);
        gridCopy(static_cast<char*>(bufs.p[dst]) + b * 16, static_cast<const char*>(bufs.p[root]) + b * 16,
                 (en - b) * 16, vec, tid, nthreads);
      }
      // Unaligned tail goes directly.
      for (size_t i = units * 16 + tid; i < bytes; i += nthreads) {
        const char c = static_cast<const char*>(bufs.p[root])[i];
        for (int r = 1; r < P; r++) static_cast<char*>(bufs.p[(root + r) % P])[i] = c;
      }
    }
    if (!blockBarrier(a, e + 2)) {
      retire(a, used, 0);
      return;
    }
    // Every rank (the root too: nobody else holds its slice) now pushes the slice it
    // owns to all ranks that still miss it, i.e. everyone but itself and the root.
    {
      size_t b, en;
      shareOf(units, P, a.rank, b, en);
      const char* src = static_cast<const char*>(bufs.p[a.rank]) + b * 16;
      const size_t nvec = vec ? (en - b) : 0;
      for (size_t v = tid; v < nvec; v += nthreads) {
        const Pack16 p = ld128_stream(src + v * 16);
        for (int i = 1; i < P; i++) {
          const int dst = (a.rank + i) % P;
          if (dst != root) st128_stream(static_cast<char*>(bufs.p[dst]) + b * 16 + v * 16, p);
        }
      }
      for (size_t i = nvec * 16 + tid; i < (en - b) * 16; i += nthreads) {
        const char c = src[i];
        for (int r = 1; r < P; r++) {
          const int dst = (a.rank + r) % P;
          if (dst != root) (static_cast<char*>(bufs.p[dst]) + b * 16)[i] = c;
        }
      }
    }
  }
  blockBarrier(a, e + used);
  retire(a, used, 0);
}

void launchBroadcast(const CommArgs& a, const PeerPtrs& bufs, void* mc, size_t bytes, int root, int mode, bool vec,
                     int blocks, int tile, cudaStream_t stream) {
  broadcastKernel<<<blocks, kThreads, 0, stream>>>(a, bufs, static_cast<char*>(mc), bytes, root, mode, vec,
                                                   tile > 0 ? tile : 1024);
}

// ---- allgather(v) / gather(v): push my block into peers' outputs ---------------------------
// Rank r's input block (inBytes[r] bytes at `in`) lands at outOff[r] in the output
// of every rank in [dstBegin, dstEnd) — all ranks for allgather, just the root for
// gather. Outputs are peer-mapped; the input is only read locally.
struct VArgs {
  size_t off[kMaxRanks];
  size_t len[kMaxRanks];
};

__global__ void __launch_bounds__(kThreads, 2)
gatherPushKernel(CommArgs a, const char* __restrict__ in, PeerPtrs outs, char* mcOut, VArgs va, int onlyDst,
                 bool vec) {
  const uint32_t e = loadEpoch(a);
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const int P = a.nranks;
  if (!blockBarrier<false>(a, e + 1)) {
    retire(a, 2, 0);
    return;
  }
  const size_t off = va.off[a.rank];
  const size_t len = va.len[a.rank];
  const bool v16 = vec && off % 16 == 0;
  const size_t nvec = v16 ? len / 16 : 0;
  if (onlyDst >= 0) {
    gridCopy(static_cast<char*>(outs.p[onlyDst]) + off, in, len, v16, tid, nthreads);
  } else if (mcOut != nullptr && v16) {
    for (size_t v = tid; v < nvec; v += nthreads) multimemSt128(mcOut + off + v * 16, ld128_stream(in + v * 16));
    for (size_t i = nvec * 16 + tid; i < len; i += nthreads) {
      const char c = in[i];
      for (int r = 0; r < P; r++) (static_cast<char*>(outs.p[r]) + off)[i] = c;
    }
  } else {
    constexpr int U = 4;
    for (size_t v0 = tid; v0 < nvec; v0 += nthreads * U) {
      Pack16 p[U];
#pragma unroll
      for (int u = 0; u < U; u++) {
        const size_t v = v0 + u * nthreads;
        if (v < nvec) p[u] = ld128_stream(in + v * 16);
      }
      for (int i = 0; i < P; i++) {
        char* dst = static_cast<char*>(outs.p[(a.rank + i) % P]) + off;
#pragma unroll
        for (int u = 0; u < U; u++) {
          const size_t v = v0 + u * nthreads;
          if (v < nvec) st128_stream(dst + v * 16, p[u]);
        }
      }
    }
    for (size_t i = nvec * 16 + tid; i < len; i += nthreads) {
      const char c = in[i];
      for (int r = 0; r < P; r++) (static_cast<char*>(outs.p[r]) + off)[i] = c;
    }
  }
  blockBarrier(a, e + 2);
  retire(a, 2, 0);
}

// Same protocol (two barriers, same CTA count) with the payload moved by the TMA: every CTA loads
// its slice of my block into shared memory ONCE (cp.async.bulk) and stores it to every peer from
// there; one thread per CTA issues, no data passes through registers.
__global__ void __launch_bounds__(128)
gatherBulkKernel(CommArgs a, const char* __restrict__ in, PeerPtrs outs, VArgs va, int onlyDst) {
  extern __shared__ __align__(128) char smem[];
  __shared__ BulkRing ring;
  bulkRingInit(ring);
  const uint32_t e = loadEpoch(a);
  const int P = a.nranks;
  if (!blockBarrier<false>(a, e + 1)) {
    retire(a, 2, 0);
    return;
  }
  const size_t off = va.off[a.rank], len = va.len[a.rank];
  const size_t units = len / 16;
  const size_t per = (units + gridDim.x - 1) / gridDim.x;
  const size_t lo = static_cast<size_t>(blockIdx.x) * per, hi = lo + per < units ? lo + per : units;
  char* dst[kMaxRanks];
  int ndst = 0;
#pragma unroll
  for (int i = 0; i < kMaxRanks; i++) {
    dst[i] = nullptr;
    if (onlyDst < 0 && i < P) dst[ndst++] = static_cast<char*>(outs.p[(a.rank + i) % P]) + off + lo * 16;
  }
  if (onlyDst >= 0) dst[ndst++] = static_cast<char*>(outs.p[onlyDst]) + off + lo * 16;
  if (lo < hi) ctaBulkCopy<kMaxRanks>(ring, smem, in + lo * 16, dst, ndst, (hi - lo) * 16);
  if (blockIdx.x == 0) {  // sub-16-byte tail
    for (size_t i = units * 16 + threadIdx.x; i < len; i += blockDim.x) {
      const char c = in[i];
      if (onlyDst >= 0) {
        (static_cast<char*>(outs.p[onlyDst]) + off)[i] = c;
      } else {
        for (int r = 0; r < P; r++) (static_cast<char*>(outs.p[r]) + off)[i] = c;
      }
    }
  }
  blockBarrier(a, e + 2);
  retire(a, 2, 0);
}

void launchGatherPush(const CommArgs& a, const void* in, const PeerPtrs& outs, void* mcOut, const size_t* offs,
                      const size_t* lens, int onlyDst, bool vec, int blocks, cudaStream_t stream, bool tma) {
  VArgs va;
  for (int i = 0; i < kMaxRanks; i++) {
    va.off[i] = i < a.nranks ? offs[i] : 0;
    va.len[i] = i < a.nranks ? lens[i] : 0;
  }
  // The TMA variant needs 16-byte aligned source, offset and destinations; a rank whose
  // pointers do not qualify runs the LDG/STG kernel with the SAME grid and barrier protocol.
  bool aligned = vec && reinterpret_cast<uintptr_t>(in) % 16 == 0 && va.off[a.rank] % 16 == 0 && mcOut == nullptr;
  for (int i = 0; i < a.nranks; i++) aligned = aligned && reinterpret_cast<uintptr_t>(outs.p[i]) % 16 == 0;
  if (tma && aligned) {
    gatherBulkKernel<<<blocks, 128, kBulkSmemBytes, stream>>>(a, static_cast<const char*>(in), outs, va, onlyDst);
    return;
  }
  gatherPushKernel<<<blocks, kThreads, 0, stream>>>(a, static_cast<const char*>(in), outs, static_cast<char*>(mcOut),
                                                    va, onlyDst, vec);
}

// ---- allgather(v) with a dtype conversion --------------------------------------------------
// Same barriers and grid rule as gatherPushKernel; offsets and lengths are in ELEMENTS. Rank r
// reads its block once as TI, converts it once (round to nearest even when narrowing, exact
// when widening) and stores it at element offset off[r] of every rank's TO output, peers
// rotated. Items of 8 elements while `in` and my output byte offset are 16-byte aligned.
template <typename TI, typename TO>
__global__ void __launch_bounds__(kThreads, 2)
gatherPushCastKernel(CommArgs a, const TI* __restrict__ in, PeerPtrs outs, VArgs va, bool vec) {
  using II = Item8<TI>;
  using OI = Item8<TO>;
  const uint32_t e = loadEpoch(a);
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const int P = a.nranks;
  if (!blockBarrier<false>(a, e + 1)) {
    retire(a, 2, 0);
    return;
  }
  const size_t off = va.off[a.rank], len = va.len[a.rank];
  const size_t outByte = off * sizeof(TO);
  const bool v16 = vec && reinterpret_cast<uintptr_t>(in) % 16 == 0 && outByte % 16 == 0;
  const size_t nitems = v16 ? len / 8 : 0;
  constexpr int U = sizeof(TI) == 4 ? 2 : 4;  // 64 bytes of input in flight per thread
  for (size_t i0 = tid; i0 < nitems; i0 += nthreads * U) {
    float v[U][8];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const size_t it = i0 + u * nthreads;
      if (it < nitems) II::load(reinterpret_cast<const char*>(in) + it * II::kBytes, v[u]);
    }
    for (int i = 0; i < P; i++) {
      char* dst = static_cast<char*>(outs.p[(a.rank + i) % P]) + outByte;
#pragma unroll
      for (int u = 0; u < U; u++) {
        const size_t it = i0 + u * nthreads;
        if (it < nitems) OI::store(dst + it * OI::kBytes, v[u]);
      }
    }
  }
  for (size_t i = nitems * 8 + tid; i < len; i += nthreads) {
    const TO o = fromAcc<TO, float>(toAcc<TI>(in[i]));
    for (int r = 0; r < P; r++) static_cast<TO*>(outs.p[(a.rank + r) % P])[off + i] = o;
  }
  blockBarrier(a, e + 2);
  retire(a, 2, 0);
}

const void* gatherPushCastKernelFor(DataType in, DataType out) {
  return dispatchCast(in, out, [](auto ti, auto to) { return fn(gatherPushCastKernel<decltype(ti), decltype(to)>); });
}

void launchGatherPushCast(const CommArgs& a, const void* in, const PeerPtrs& outs, const size_t* elemOff,
                          const size_t* elemLen, DataType dt, DataType outDt, bool vec, int blocks,
                          cudaStream_t stream) {
  const void* k = gatherPushCastKernelFor(dt, outDt);
  if (k == nullptr) return;
  VArgs va;
  for (int i = 0; i < kMaxRanks; i++) {
    va.off[i] = i < a.nranks ? elemOff[i] : 0;
    va.len[i] = i < a.nranks ? elemLen[i] : 0;
  }
  CommArgs ca = a;
  PeerPtrs po = outs;
  void* args[] = {&ca, &in, &po, &va, &vec};
  launchKernel(k, blocks, kThreads, args, stream);
}

// ---- alltoall(v) / scatter: push chunk j of my input into slot (me) of rank j's output -------
// sendOff/sendLen index my input per destination; recvOff[r] (same on all ranks by
// symmetry of the exchange tables) is where MY chunk lands in rank r's output.
__global__ void __launch_bounds__(kThreads)
alltoallPushKernel(CommArgs a, const char* __restrict__ in, PeerPtrs outs, VArgs send, VArgs dstOff, VArgs myRecv,
                   VArgs blk, bool exchange, int onlySrc, bool vec) {
  const uint32_t e = loadEpoch(a);
  const int P = a.nranks;
  // v-variant: publish where I expect each source's chunk; peers read it after the
  // barrier (every CTA writes the same values, so no cross-CTA ordering is needed).
  if (exchange && threadIdx.x < P) a.self->xchg[threadIdx.x] = myRecv.off[threadIdx.x];
  if (!blockBarrier(a, e + 1)) {
    retire(a, 2, 0);
    return;
  }
  if (onlySrc < 0 || onlySrc == a.rank) {
    // CTAs are dealt to destinations in proportion to the bytes each one gets (the host
    // fills blk.off = first CTA, blk.len = CTA count per destination), so every link is
    // busy at once and uneven (v-variant) splits stay balanced. With fewer CTAs than
    // destinations every CTA walks all destinations.
    const bool partitioned = blk.len[0] + blk.off[P - 1] > 0 && static_cast<size_t>(gridDim.x) >= static_cast<size_t>(P);
    for (int i = 0; i < P; i++) {
      const int dst = (a.rank + i) % P;
      size_t tid, nthreads;
      if (partitioned) {
        const size_t b0 = blk.off[dst], nb = blk.len[dst];
        if (blockIdx.x < b0 || blockIdx.x >= b0 + nb) continue;
        tid = (blockIdx.x - b0) * blockDim.x + threadIdx.x;
        nthreads = nb * blockDim.x;
      } else {
        tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
        nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
      }
      const size_t so = send.off[dst], sl = send.len[dst];
      const size_t dofs = exchange ? static_cast<size_t>(*reinterpret_cast<volatile unsigned long long*>(
                                         &a.sig[dst]->xchg[a.rank]))
                                   : dstOff.off[dst];
      gridCopy(static_cast<char*>(outs.p[dst]) + dofs, in + so, sl, vec, tid, nthreads);
    }
  }
  blockBarrier(a, e + 2);
  retire(a, 2, 0);
}

void launchAlltoallPush(const CommArgs& a, const void* in, const PeerPtrs& outs, const size_t* sendOff,
                        const size_t* sendLen, const size_t* dstOff, const size_t* recvOffTable, int onlySrc,
                        bool vec, int blocks, cudaStream_t stream) {
  VArgs s, d, rcv;
  for (int i = 0; i < kMaxRanks; i++) {
    s.off[i] = i < a.nranks ? sendOff[i] : 0;
    s.len[i] = i < a.nranks ? sendLen[i] : 0;
    d.off[i] = i < a.nranks ? dstOff[i] : 0;
    d.len[i] = 0;
    rcv.off[i] = (recvOffTable != nullptr && i < a.nranks) ? recvOffTable[i] : 0;
    rcv.len[i] = 0;
  }
  // CTA ranges per destination, proportional to payload (at least one each).
  VArgs blk;
  for (int i = 0; i < kMaxRanks; i++) blk.off[i] = blk.len[i] = 0;
  if (blocks >= a.nranks) {
    size_t total = 0;
    for (int i = 0; i < a.nranks; i++) total += s.len[i];
    size_t used = 0;
    int spare = blocks - a.nranks;
    for (int i = 0; i < a.nranks; i++) {
      size_t extra = total > 0 ? static_cast<size_t>(spare) * s.len[i] / total : 0;
      blk.off[i] = used;
      blk.len[i] = 1 + extra;
      used += blk.len[i];
    }
  }
  alltoallPushKernel<<<blocks, kThreads, 0, stream>>>(a, static_cast<const char*>(in), outs, s, d, rcv, blk,
                                                      recvOffTable != nullptr, onlySrc, vec);
}

// ---- reduce_scatter / reduce: pull my slice from every peer's input, reduce, store -----------
// Inputs are peer-mapped. Rank r reduces elements [elemOff[r], elemOff[r]+elemLen[r])
// and writes them to `out` (local pointer; for reduce() it is the root's peer-mapped
// output at the same offset).
struct EArgs {
  size_t off[kMaxRanks];
  size_t len[kMaxRanks];
};

template <typename T, int NR, int UNROLL>
__global__ void __launch_bounds__(kThreads)
reducePullKernel(CommArgs a, PeerPtrs ins, char* mcIn, T* __restrict__ out, EArgs ea, DevOp op, float scale,
                 bool vec, bool useMc) {
  using PT = PackTraits<T>;
  const uint32_t e = loadEpoch(a);
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const int P = NR > 0 ? NR : a.nranks;
  if (!blockBarrier<false>(a, e + 1)) {
    retire(a, 2, 0);
    return;
  }
  const size_t off = ea.off[a.rank], len = ea.len[a.rank];
  const bool v16 = vec && (off * sizeof(T)) % 16 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0;
  const size_t nvec = v16 ? len / PT::kElems : 0;
  const size_t byteOff = off * sizeof(T);
  if (useMc && v16) {
    if constexpr (isHotType<T>()) {
      constexpr int U = 4;
      for (size_t v0 = tid; v0 < nvec; v0 += nthreads * U) {
        Pack16 r[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
          const size_t v = v0 + u * nthreads;
          if (v < nvec) r[u] = Multimem<T>::ldReduceAdd(mcIn + byteOff + v * 16);
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
          const size_t v = v0 + u * nthreads;
          if (v < nvec) {
            if (scale != 1.0f) r[u] = scalePack<T>(r[u], scale);
            st128(reinterpret_cast<char*>(out) + v * 16, r[u]);
          }
        }
      }
    }
  } else {
    constexpr int kSlots = NR > 0 ? NR : kMaxRanks;
    const char* peer[kSlots];
#pragma unroll
    for (int i = 0; i < kSlots; i++) {
      peer[i] = i < P ? static_cast<const char*>(ins.p[(a.rank + i) % P]) + byteOff : nullptr;
    }
    for (size_t v0 = tid; v0 < nvec; v0 += nthreads * UNROLL) {
      Pack16 p[UNROLL][kSlots];
#pragma unroll
      for (int u = 0; u < UNROLL; u++) {
        const size_t v = v0 + static_cast<size_t>(u) * nthreads;
        if (v < nvec) {
#pragma unroll
          for (int i = 0; i < kSlots; i++) {
            if (i < P) p[u][i] = ld128_stream(peer[i] + v * 16);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < UNROLL; u++) {
        const size_t v = v0 + static_cast<size_t>(u) * nthreads;
        if (v < nvec) {
          typename PT::AccPack acc = PT::widen(p[u][0]);
#pragma unroll
          for (int i = 1; i < kSlots; i++) {
            if (i < P) PT::combine(acc, p[u][i], op);
          }
          if (scale != 1.0f) PT::scale(acc, scale);
          st128(reinterpret_cast<char*>(out) + v * 16, PT::narrow(acc));
        }
      }
    }
  }
  for (size_t i = nvec * PT::kElems + tid; i < len; i += nthreads) {
    using A = typename AccType<T>::type;
    A acc = toAcc<T>(static_cast<const T*>(ins.p[0])[off + i]);
    for (int r = 1; r < P; r++) acc = applyOp<A>(acc, toAcc<T>(static_cast<const T*>(ins.p[r])[off + i]), op);
    if (scale != 1.0f) acc = scaleAcc(acc, scale);
    out[i] = fromAcc<T, A>(acc);
  }
  blockBarrier(a, e + 2);
  retire(a, 2, 0);
}

namespace {
// The instantiation of the reduce pull kernel for (T, P): rank-count specialisations of the
// hot types with their unroll, the generic kernel otherwise.
template <typename T>
const void* reducePullFn(int P) {
  if constexpr (isHotType<T>()) {
    if (P == 2) return fn(reducePullKernel<T, 2, 4>);
    if (P == 4) return fn(reducePullKernel<T, 4, 2>);
    if (P == 8) return fn(reducePullKernel<T, 8, 2>);
  }
  return fn(reducePullKernel<T, 0, 1>);
}
}  // namespace

const void* reducePullKernelPtr(DataType dt, int nranks) {
  return dispatchType(dt, [&](auto t) { return reducePullFn<decltype(t)>(nranks); });
}

void launchReducePull(const CommArgs& a, const PeerPtrs& ins, void* mcIn, void* out, const size_t* elemOff,
                      const size_t* elemLen, DataType dt, ReduceOp op, float scale, bool vec, bool useMc, int blocks,
                      cudaStream_t stream) {
  EArgs ea;
  for (int i = 0; i < kMaxRanks; i++) {
    ea.off[i] = i < a.nranks ? elemOff[i] : 0;
    ea.len[i] = i < a.nranks ? elemLen[i] : 0;
  }
  CommArgs ca = a;
  PeerPtrs pi = ins;
  char* mc = static_cast<char*>(mcIn);
  DevOp dop = static_cast<DevOp>(op);
  void* args[] = {&ca, &pi, &mc, &out, &ea, &dop, &scale, &vec, &useMc};
  launchKernel(reducePullKernelPtr(dt, a.nranks), blocks, kThreads, args, stream);
}

// ---- reduce_scatter with a dtype conversion --------------------------------------------------
// Same barriers, CTA pairing and share tables as reducePullKernel. Rank r pulls its share of
// every peer's TI input in rank-rotated order, accumulates in fp32, applies `scale` to the
// accumulator, rounds once to TO and stores to its local `out`. Items of 8 elements while my
// input byte offset and `out` are 16-byte aligned; the rank-count specialisations load every
// peer's item before reducing any (UNROLL items per thread), as reducePullKernel does. It never uses
// multimem.ld_reduce: the switch returns the input dtype, so a 16-bit input would be rounded
// to 16 bits before the fp32 result is formed.
template <typename TI, typename TO, int NR, int UNROLL>
__global__ void __launch_bounds__(kThreads, 1)
reducePullCastKernel(CommArgs a, PeerPtrs ins, TO* __restrict__ out, EArgs ea, DevOp op, float scale, bool vec) {
  using II = Item8<TI>;
  using OI = Item8<TO>;
  constexpr int kPk = II::kPacks;
  const uint32_t e = loadEpoch(a);
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const int P = NR > 0 ? NR : a.nranks;
  if (!blockBarrier<false>(a, e + 1)) {
    retire(a, 2, 0);
    return;
  }
  const size_t off = ea.off[a.rank], len = ea.len[a.rank];
  const size_t byteOff = off * sizeof(TI);
  const bool v16 = vec && byteOff % 16 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0;
  const size_t nitems = v16 ? len / 8 : 0;
  if constexpr (NR > 0) {
    const char* peer[NR];
#pragma unroll
    for (int i = 0; i < NR; i++) peer[i] = static_cast<const char*>(ins.p[(a.rank + i) % NR]) + byteOff;
    for (size_t i0 = tid; i0 < nitems; i0 += nthreads * UNROLL) {
      Pack16 p[UNROLL][NR][kPk];
#pragma unroll
      for (int u = 0; u < UNROLL; u++) {
        const size_t it = i0 + static_cast<size_t>(u) * nthreads;
        if (it < nitems) {
#pragma unroll
          for (int i = 0; i < NR; i++) {
#pragma unroll
            for (int k = 0; k < kPk; k++) p[u][i][k] = ld128_stream(peer[i] + it * II::kBytes + k * 16);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < UNROLL; u++) {
        const size_t it = i0 + static_cast<size_t>(u) * nthreads;
        if (it < nitems) {
          float acc[8];
          II::widen(p[u][0], acc);
#pragma unroll
          for (int i = 1; i < NR; i++) {
            float x[8];
            II::widen(p[u][i], x);
#pragma unroll
            for (int k = 0; k < 8; k++) acc[k] = applyOp<float>(acc[k], x[k], op);
          }
          if (scale != 1.0f) {
#pragma unroll
            for (int k = 0; k < 8; k++) acc[k] *= scale;
          }
          OI::template store<false>(reinterpret_cast<char*>(out) + it * OI::kBytes, acc);
        }
      }
    }
  } else {
    // Any rank count: one peer's item at a time.
    for (size_t it = tid; it < nitems; it += nthreads) {
      float acc[8];
      II::load(static_cast<const char*>(ins.p[a.rank]) + byteOff + it * II::kBytes, acc);
      for (int i = 1; i < P; i++) {
        float x[8];
        II::load(static_cast<const char*>(ins.p[(a.rank + i) % P]) + byteOff + it * II::kBytes, x);
#pragma unroll
        for (int k = 0; k < 8; k++) acc[k] = applyOp<float>(acc[k], x[k], op);
      }
      if (scale != 1.0f) {
#pragma unroll
        for (int k = 0; k < 8; k++) acc[k] *= scale;
      }
      OI::template store<false>(reinterpret_cast<char*>(out) + it * OI::kBytes, acc);
    }
  }
  for (size_t i = nitems * 8 + tid; i < len; i += nthreads) {
    float acc = toAcc<TI>(static_cast<const TI*>(ins.p[a.rank])[off + i]);
    for (int r = 1; r < P; r++) {
      acc = applyOp<float>(acc, toAcc<TI>(static_cast<const TI*>(ins.p[(a.rank + r) % P])[off + i]), op);
    }
    if (scale != 1.0f) acc = scaleAcc(acc, scale);
    out[i] = fromAcc<TO, float>(acc);
  }
  blockBarrier(a, e + 2);
  retire(a, 2, 0);
}

namespace {
// The instantiation for (TI, TO, P): rank-count specialisations with the unroll of
// reducePullFn for 16-bit inputs, half of it for f32 inputs (twice the bytes per item), so
// both keep the same bytes in flight per thread as the same-dtype pull kernel.
template <typename TI, typename TO>
const void* reducePullCastFn(int P) {
  constexpr int W = sizeof(TI) == 4 ? 2 : 1;
  if (P == 2) return fn(reducePullCastKernel<TI, TO, 2, 4 / W>);
  if (P == 4) return fn(reducePullCastKernel<TI, TO, 4, 2 / W>);
  if (P == 8) return fn(reducePullCastKernel<TI, TO, 8, 2 / W>);
  return fn(reducePullCastKernel<TI, TO, 0, 1>);
}
}  // namespace

const void* reducePullCastKernelFor(DataType in, DataType out, int nranks) {
  return dispatchCast(in, out, [&](auto ti, auto to) { return reducePullCastFn<decltype(ti), decltype(to)>(nranks); });
}

void launchReducePullCast(const CommArgs& a, const PeerPtrs& ins, void* out, const size_t* elemOff,
                          const size_t* elemLen, DataType dt, DataType outDt, ReduceOp op, float scale, bool vec,
                          int blocks, cudaStream_t stream) {
  const void* k = reducePullCastKernelFor(dt, outDt, a.nranks);
  if (k == nullptr) return;
  EArgs ea;
  for (int i = 0; i < kMaxRanks; i++) {
    ea.off[i] = i < a.nranks ? elemOff[i] : 0;
    ea.len[i] = i < a.nranks ? elemLen[i] : 0;
  }
  CommArgs ca = a;
  PeerPtrs pi = ins;
  DevOp dop = static_cast<DevOp>(op);
  void* args[] = {&ca, &pi, &out, &ea, &dop, &scale, &vec};
  launchKernel(k, blocks, kThreads, args, stream);
}


// ---- small allgather / alltoall without a barrier: flag-in-data lines -------------------------
// Same protocol and pool region as llAllreduceKernel (every rank hears from every peer in a
// launch, which is what makes two parity halves sufficient). Payload unit: 8 bytes.
namespace {
__device__ __forceinline__ void load8(const char* p, size_t avail, bool aligned, uint32_t& d0, uint32_t& d1) {
  if (aligned && avail >= 8) {
    const uint2 v = *reinterpret_cast<const uint2*>(p);
    d0 = v.x;
    d1 = v.y;
    return;
  }
  unsigned long long w = 0;
  for (int k = 0; k < 8; k++) {
    if (static_cast<size_t>(k) < avail) w |= static_cast<unsigned long long>(static_cast<unsigned char>(p[k])) << (8 * k);
  }
  d0 = static_cast<uint32_t>(w);
  d1 = static_cast<uint32_t>(w >> 32);
}
__device__ __forceinline__ void store8(char* p, size_t avail, bool aligned, uint32_t d0, uint32_t d1) {
  if (aligned && avail >= 8) {
    *reinterpret_cast<uint2*>(p) = make_uint2(d0, d1);
    return;
  }
  const unsigned long long w = static_cast<unsigned long long>(d0) | (static_cast<unsigned long long>(d1) << 32);
  for (int k = 0; k < 8; k++) {
    if (static_cast<size_t>(k) < avail) p[k] = static_cast<char>(w >> (8 * k));
  }
}
}  // namespace

__global__ void __launch_bounds__(kThreads)
llExchangeKernel(CommArgs a, const char* __restrict__ in, char* __restrict__ out, size_t bytes, int mode, PeerPtrs ll,
                 size_t srcStride, size_t parityStride) {
  const uint32_t seq = ld_relaxed_sys(&a.self->llSeq) + 1u;
  const size_t base = (seq & 1u) * parityStride;
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const int P = a.nranks;
  const size_t nunits = (bytes + 7) / 8;
  const size_t items = static_cast<size_t>(P) * nunits;
  const bool inAligned = reinterpret_cast<uintptr_t>(in) % 8 == 0 && bytes % 8 == 0;
  const bool outAligned = reinterpret_cast<uintptr_t>(out) % 8 == 0 && bytes % 8 == 0;
  // send: item = (peer slot i, unit u); peers rotated by rank
  for (size_t it = tid; it < items; it += nthreads) {
    const int i = static_cast<int>(it / nunits);
    const size_t u = it % nunits;
    const int dst = (a.rank + i) % P;
    const char* src = in + (mode == 1 ? static_cast<size_t>(dst) * bytes : 0) + u * 8;
    uint32_t d0, d1;
    load8(src, bytes - u * 8, inAligned, d0, d1);
    if (dst == a.rank) {
      store8(out + static_cast<size_t>(a.rank) * bytes + u * 8, bytes - u * 8, outAligned, d0, d1);
    } else {
      llStore(static_cast<char*>(ll.p[dst]) + base + static_cast<size_t>(a.rank) * srcStride + u * 16, d0, d1, seq);
    }
  }
  // receive
  const char* mine = static_cast<const char*>(ll.p[a.rank]) + base;
  for (size_t it = tid; it < items; it += nthreads) {
    const int i = static_cast<int>(it / nunits);
    const size_t u = it % nunits;
    const int src = (a.rank + i) % P;
    if (src == a.rank) continue;
    uint32_t d0, d1;
    if (!llLoad(a, mine + static_cast<size_t>(src) * srcStride + u * 16, seq, d0, d1, src)) break;
    store8(out + static_cast<size_t>(src) * bytes + u * 8, bytes - u * 8, outAligned, d0, d1);
  }
  retire(a, 0, 0, 1);
}

void launchLLExchange(const CommArgs& a, const void* in, void* out, size_t bytes, int mode, const PeerPtrs& ll,
                      size_t srcStride, size_t parityStride, int blocks, int threads, cudaStream_t stream) {
  llExchangeKernel<<<blocks, threads, 0, stream>>>(a, static_cast<const char*>(in), static_cast<char*>(out), bytes, mode,
                                                   ll, srcStride, parityStride);
}

const void* broadcastKernelPtr() { return fn(broadcastKernel); }
const void* gatherPushKernelPtr() { return fn(gatherPushKernel); }
const void* gatherBulkKernelPtr() { return fn(gatherBulkKernel); }
const void* alltoallPushKernelPtr() { return fn(alltoallPushKernel); }

void preloadCollectiveKernels() {
  touch(fn(broadcastKernel));
  touch(fn(gatherPushKernel));
  cudaFuncSetAttribute(fn(gatherBulkKernel), cudaFuncAttributeMaxDynamicSharedMemorySize,
                       static_cast<int>(kBulkSmemBytes));
  touch(fn(gatherBulkKernel));
  touch(fn(alltoallPushKernel));
  touch(fn(llExchangeKernel));
  for (DataType dt : kAllDataTypes) {
    for (int P : {0, 2, 4, 8}) touch(reducePullKernelPtr(dt, P));
    for (DataType outDt : kAllDataTypes) {
      touch(gatherPushCastKernelFor(dt, outDt));
      for (int P : {0, 2, 4, 8}) touch(reducePullCastKernelFor(dt, outDt, P));
    }
  }
  cudaGetLastError();
}

}  // namespace cuda
}  // namespace glb
