// Point-to-point transfers between two GPUs over NVLink peer memory (sm_100a).
//
// The reference moves GPU buffers between two ranks only through a transport::Pair
// (ibverbs + GPUDirect: transport/ibverbs/pair.cc:328-384, buffer.cc:24-59) — there is no
// NVLink path. Here a send is a kernel on the sender that streams the payload into a
// mailbox ring inside the RECEIVER's symmetric pool and a recv is a kernel on the receiver
// that drains it; the two sides synchronise per chunk through head / tail counters in each
// other's signal pads (st.release.sys / ld.acquire.sys), so a transfer larger than the ring
// flows through it while both kernels run. Matching is by posting order per (src, dst)
// pair, like a connected Pair with a single slot. One kernel can play both roles
// (send to `dst` while receiving from `src`): that is what a ring exchange or a pipeline
// stage posts, and it cannot deadlock on stream order.
//
// Also here: the whole-grid copy kernel behind the one-sided put / get on peer-mapped
// memory (RemoteKey semantics, transport/unbound_buffer.h:128-152).
#include "glb/cuda/bulk_copy.cuh"
#include "glb/cuda/device_common.cuh"
#include "glb/cuda/dispatch.cuh"
#include "glb/cuda/kernels.h"

namespace glb {
namespace cuda {

namespace {

// Copy [0, bytes) with one CTA; 128-bit when both sides allow it.
__device__ __forceinline__ void ctaCopy(char* dst, const char* src, size_t bytes) {
  const uintptr_t both = reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src);
  if (both % 16 == 0) {
    const size_t nvec = bytes / 16;
    constexpr int U = 4;
    for (size_t v0 = threadIdx.x; v0 < nvec; v0 += static_cast<size_t>(blockDim.x) * U) {
      Pack16 p[U];
#pragma unroll
      for (int u = 0; u < U; u++) {
        const size_t v = v0 + static_cast<size_t>(u) * blockDim.x;
        if (v < nvec) p[u] = ld128_stream(src + v * 16);
      }
#pragma unroll
      for (int u = 0; u < U; u++) {
        const size_t v = v0 + static_cast<size_t>(u) * blockDim.x;
        if (v < nvec) st128_stream(dst + v * 16, p[u]);
      }
    }
    for (size_t i = nvec * 16 + threadIdx.x; i < bytes; i += blockDim.x) dst[i] = src[i];
  } else if (both % 4 == 0) {
    const size_t n = bytes / 4;
    for (size_t i = threadIdx.x; i < n; i += blockDim.x) {
      reinterpret_cast<unsigned int*>(dst)[i] = reinterpret_cast<const unsigned int*>(src)[i];
    }
    for (size_t i = n * 4 + threadIdx.x; i < bytes; i += blockDim.x) dst[i] = src[i];
  } else {
    for (size_t i = threadIdx.x; i < bytes; i += blockDim.x) dst[i] = src[i];
  }
}

// Block-wide wait on a counter; false when the wait was abandoned (time-out / abort).
__device__ __forceinline__ bool ctaWait(const CommArgs& a, const uint32_t* flag, uint32_t want, int peer) {
  int ok = 1;
  if (threadIdx.x == 0) {
    ok = waitFlag(a, flag, want, peer) ? 1 : 0;
  }
  return __syncthreads_and(ok) != 0;
}

}  // namespace

// Mailbox layout in every rank's pool: box[src] = nslots slots of slotBytes, each slot cut
// into `lanes` stripes (lane l of the sender fills stripe l, lane l of the receiver drains it).
// gridDim.x = sendLanes + recvLanes; the first sendLanes CTAs send.
__global__ void __launch_bounds__(kThreads)
p2pKernel(CommArgs a, const char* sendPtr, size_t sendBytes, int dst, char* recvPtr, size_t recvBytes, int src,
          PeerPtrs mailbox, size_t boxStride, size_t slotBytes, int nslots, int lanes, int sendLanes) {
  SignalPad* me = a.self;
  const size_t stripe = slotBytes / static_cast<size_t>(lanes) / 16 * 16;
  const size_t chunkBytes = stripe * lanes;
  if (static_cast<int>(blockIdx.x) < sendLanes) {
    const int l = blockIdx.x;
    const size_t nchunks = (sendBytes + chunkBytes - 1) / chunkBytes;
    uint32_t c = me->p2pSent[l][dst];
    const uint32_t* tail = &me->p2pTail[l][dst];
    uint32_t* head = &a.sig[dst]->p2pHead[l][a.rank];
    char* box = static_cast<char*>(mailbox.p[dst]) + static_cast<size_t>(a.rank) * boxStride;
    bool ok = true;
    for (size_t k = 0; k < nchunks && ok; k++, c++) {
      // the slot is free once the receiver has consumed chunk c - nslots
      if (c + 1u > static_cast<uint32_t>(nslots)) ok = ctaWait(a, tail, c + 1u - static_cast<uint32_t>(nslots), dst);
      if (!ok) break;
      const size_t lo = k * chunkBytes + static_cast<size_t>(l) * stripe;
      if (lo < sendBytes) {
        const size_t n = sendBytes - lo < stripe ? sendBytes - lo : stripe;
        ctaCopy(box + static_cast<size_t>(c % nslots) * slotBytes + static_cast<size_t>(l) * stripe, sendPtr + lo, n);
      }
      __syncthreads();
      if (threadIdx.x == 0) st_release_sys(head, c + 1u);
    }
    if (threadIdx.x == 0) me->p2pSent[l][dst] = c;
  } else {
    const int l = blockIdx.x - sendLanes;
    const size_t nchunks = (recvBytes + chunkBytes - 1) / chunkBytes;
    uint32_t c = me->p2pRecvd[l][src];
    const uint32_t* head = &me->p2pHead[l][src];
    uint32_t* tail = &a.sig[src]->p2pTail[l][a.rank];
    const char* box = static_cast<const char*>(mailbox.p[a.rank]) + static_cast<size_t>(src) * boxStride;
    bool ok = true;
    for (size_t k = 0; k < nchunks && ok; k++, c++) {
      ok = ctaWait(a, head, c + 1u, src);
      if (!ok) break;
      const size_t lo = k * chunkBytes + static_cast<size_t>(l) * stripe;
      if (lo < recvBytes) {
        const size_t n = recvBytes - lo < stripe ? recvBytes - lo : stripe;
        ctaCopy(recvPtr + lo, box + static_cast<size_t>(c % nslots) * slotBytes + static_cast<size_t>(l) * stripe, n);
      }
      __syncthreads();
      if (threadIdx.x == 0) st_release_sys(tail, c + 1u);
    }
    if (threadIdx.x == 0) me->p2pRecvd[l][src] = c;
  }
}

// ---- zero-copy neighbour exchange ----------------------------------------------------------------
// sendrecv() above costs two passes (sender -> mailbox, mailbox -> user buffer) and a flag
// round trip per 32 KB stripe: 73-100 GB/s measured on B200 against a ~690 GB/s link. When
// the RECEIVE buffer is peer-mapped (a registered / symmetric buffer that every rank uses at
// the same offset - the double-buffered K/V block of ring attention, a pipeline stage's
// activation slot) the sender can write straight into it. What is left of the protocol is
// one "ready" flag (receiver -> sender: my kernel has started, so everything that read the
// buffer earlier on my stream is done) and one arrival counter (sender CTAs -> receiver).
// Lane kXchgLane of the p2p counters carries both, lane kXchgTicket the retire ticket.
constexpr int kXchgLane = kP2pLanes - 1;
constexpr int kXchgTicket = kP2pLanes - 2;

template <bool kBulk>
__global__ void __launch_bounds__(kBulk ? 128 : kThreads)
exchangeKernel(CommArgs a, const char* sendPtr, size_t sendBytes, int dst, char* remote, size_t recvBytes, int src) {
  extern __shared__ __align__(128) char smem[];
  __shared__ BulkRing ring;
  SignalPad* me = a.self;
  // counters only change when the LAST CTA retires, after every CTA has read them
  const uint32_t sent = sendBytes ? me->p2pSent[kXchgLane][dst] : 0u;
  const uint32_t recvd = recvBytes ? me->p2pRecvd[kXchgLane][src] : 0u;
  if (recvBytes && blockIdx.x == 0 && threadIdx.x == 0) {
    st_release_sys(&a.sig[src]->p2pTail[kXchgLane][a.rank], recvd + 1u);
  }
  if (kBulk) bulkRingInit(ring);
  bool ok = true;
  if (sendBytes) {
    ok = ctaWait(a, &me->p2pTail[kXchgLane][dst], sent + 1u, dst);
    if (ok) {
      const size_t units = sendBytes / 16;
      const size_t per = (units + gridDim.x - 1) / gridDim.x;
      const size_t lo = static_cast<size_t>(blockIdx.x) * per, hi = lo + per < units ? lo + per : units;
      if (lo < hi) {
        if (kBulk) {
          char* const d[1] = {remote + lo * 16};
          ctaBulkCopy<1>(ring, smem, sendPtr + lo * 16, d, 1, (hi - lo) * 16);
        } else {
          ctaCopy(remote + lo * 16, sendPtr + lo * 16, (hi - lo) * 16);
        }
      }
      if (blockIdx.x == gridDim.x - 1) {
        for (size_t i = units * 16 + threadIdx.x; i < sendBytes; i += blockDim.x) remote[i] = sendPtr[i];
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        __threadfence_system();
        atomicAdd_system(&a.sig[dst]->p2pHead[kXchgLane][a.rank], 1u);
      }
    }
  }
  if (recvBytes && ok) ok = ctaWait(a, &me->p2pHead[kXchgLane][src], (recvd + 1u) * gridDim.x, src);
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t* ticket = sendBytes ? &me->p2pSent[kXchgTicket][dst] : &me->p2pRecvd[kXchgTicket][src];
    if (atomicAdd(ticket, 1u) == gridDim.x - 1) {
      *ticket = 0u;
      if (sendBytes) me->p2pSent[kXchgLane][dst] = sent + 1u;
      if (recvBytes) me->p2pRecvd[kXchgLane][src] = recvd + 1u;
    }
  }
}

__global__ void __launch_bounds__(kThreads) peerCopyKernel(char* dst, const char* src, size_t bytes) {
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const size_t nthreads = static_cast<size_t>(gridDim.x) * blockDim.x;
  const uintptr_t both = reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src);
  if (both % 16 == 0) {
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
        if (v < nvec) st128_stream(dst + v * 16, p[u]);
      }
    }
    for (size_t i = nvec * 16 + tid; i < bytes; i += nthreads) dst[i] = src[i];
  } else {
    for (size_t i = tid; i < bytes; i += nthreads) dst[i] = src[i];
  }
}

// put / get through the TMA: every CTA streams one contiguous slice (one issuing thread).
__global__ void __launch_bounds__(128) peerBulkCopyKernel(char* dst, const char* src, size_t bytes) {
  extern __shared__ __align__(128) char smem[];
  __shared__ BulkRing ring;
  bulkRingInit(ring);
  const size_t units = bytes / 16;
  const size_t per = (units + gridDim.x - 1) / gridDim.x;
  const size_t lo = static_cast<size_t>(blockIdx.x) * per, hi = lo + per < units ? lo + per : units;
  if (lo < hi) {
    char* const d[1] = {dst + lo * 16};
    ctaBulkCopy<1>(ring, smem, src + lo * 16, d, 1, (hi - lo) * 16);
  }
  if (blockIdx.x == 0) {
    for (size_t i = units * 16 + threadIdx.x; i < bytes; i += blockDim.x) dst[i] = src[i];
  }
}

void preloadP2pKernels() {
  cudaFuncSetAttribute(fn(peerBulkCopyKernel), cudaFuncAttributeMaxDynamicSharedMemorySize,
                       static_cast<int>(kBulkSmemBytes));
  touch(fn(p2pKernel));
  touch(fn(peerCopyKernel));
  touch(fn(peerBulkCopyKernel));
  touch(fn(exchangeKernel<false>));
  touch(fn(exchangeKernel<true>));
  cudaFuncSetAttribute(fn(exchangeKernel<true>), cudaFuncAttributeMaxDynamicSharedMemorySize, kBulkSmemBytes);
  cudaGetLastError();
}

void launchP2p(const CommArgs& a, const void* sendPtr, size_t sendBytes, int dst, void* recvPtr, size_t recvBytes,
               int src, const PeerPtrs& mailbox, size_t boxStride, size_t slotBytes, int nslots, int lanes,
               cudaStream_t stream) {
  const int sendLanes = sendBytes > 0 ? lanes : 0;
  const int recvLanes = recvBytes > 0 ? lanes : 0;
  if (sendLanes + recvLanes == 0) return;
  p2pKernel<<<sendLanes + recvLanes, kThreads, 0, stream>>>(a, static_cast<const char*>(sendPtr), sendBytes, dst,
                                                            static_cast<char*>(recvPtr), recvBytes, src, mailbox,
                                                            boxStride, slotBytes, nslots, lanes, sendLanes);
}

void launchExchange(const CommArgs& a, const void* sendPtr, size_t sendBytes, int dst, void* remote, size_t recvBytes,
                    int src, int blocks, bool tma, cudaStream_t stream) {
  const bool aligned = (reinterpret_cast<uintptr_t>(remote) | reinterpret_cast<uintptr_t>(sendPtr)) % 16 == 0;
  if (tma && (aligned || sendBytes == 0)) {
    exchangeKernel<true><<<blocks, 128, kBulkSmemBytes, stream>>>(a, static_cast<const char*>(sendPtr), sendBytes, dst,
                                                                 static_cast<char*>(remote), recvBytes, src);
  } else {
    exchangeKernel<false><<<blocks, kThreads, 0, stream>>>(a, static_cast<const char*>(sendPtr), sendBytes, dst,
                                                          static_cast<char*>(remote), recvBytes, src);
  }
}

void launchPeerCopy(void* dst, const void* src, size_t bytes, int blocks, cudaStream_t stream, bool tma) {
  if (bytes == 0) return;
  const bool aligned = (reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) % 16 == 0;
  if (tma && aligned && bytes >= 64 * 1024) {
    peerBulkCopyKernel<<<blocks, 128, kBulkSmemBytes, stream>>>(static_cast<char*>(dst), static_cast<const char*>(src), bytes);
  } else {
    peerCopyKernel<<<blocks, kThreads, 0, stream>>>(static_cast<char*>(dst), static_cast<const char*>(src), bytes);
  }
}

}  // namespace cuda
}  // namespace glb
