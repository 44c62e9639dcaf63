// Host-callable launchers for the device kernels (implemented in the .cu files).
#pragma once

#include <cuda_runtime.h>

#include "glb/cuda/comm_types.h"
#include "glb/types.h"

namespace glb {
namespace cuda {

// Force-load all kernels of the library on the current device (idempotent, cheap).
void preloadAllreduceKernels();
void preloadCollectiveKernels();
void preloadScheduleKernels();
void preloadLocalKernels();
void preloadPipelineKernels();
void preloadP2pKernels();

// allreduce_kernels.cu ---------------------------------------------------------------------
void launchBarrier(const CommArgs& a, cudaStream_t stream);
// Flag-in-data one-shot (no barrier). `ll.p[r]` = LL region of rank r's pool.
void launchLLAllreduce(const CommArgs& a, const void* in, void* out, size_t count, DataType dt, DataType outDt,
                       ReduceOp op, float scale, const PeerPtrs& ll, size_t srcStride, size_t parityStride,
                       const LocalPtrs& extra, int blocks, int threads, cudaStream_t stream);
// Small reduce_scatter (equal shares of `perRank` elements), flag-in-data, no barrier.
void launchLLReduceScatter(const CommArgs& a, const void* in, void* out, size_t perRank, DataType dt, ReduceOp op,
                           float scale, const PeerPtrs& ll, size_t srcStride, size_t parityStride, int blocks, int threads,
                           cudaStream_t stream);
void launchOneShotAllreduce(const CommArgs& a, const void* in, void* out, size_t count, DataType dt, ReduceOp op,
                            float scale, const PeerPtrs& stage, size_t halfBytes, const LocalPtrs& extra, int blocks,
                            cudaStream_t stream);
void launchTwoShotAllreduce(const CommArgs& a, const PeerPtrs& bufs, size_t count, DataType dt, ReduceOp op,
                            float scale, bool vectorOk, const LocalPtrs& extra, const LaunchCfg& cfg,
                            cudaStream_t stream);
bool nvlsSupports(DataType dt, ReduceOp op);
void setOneShotPush(bool on);  // tuning / A-B testing of the push flavour of one-shot
bool oneShotPushEnabled();
void launchNvlsAllreduce(const CommArgs& a, void* mcPtr, const PeerPtrs& bufs, size_t count, DataType dt, float scale,
                         const LocalPtrs& extra, const LaunchCfg& cfg, cudaStream_t stream);
// NVLS on the first part of the vector + peer-to-peer two-shot on the rest, concurrently
// (P = 4 or 8, sum of f32 / f16 / bf16, multicast-bound buffer).
const void* hybridKernelFor(DataType dt, int nranks);
void launchHybridAllreduce(const CommArgs& a, void* mcPtr, const PeerPtrs& bufs, size_t count, DataType dt, float scale,
                           int blocks, int nvlsBlocks, unsigned p2pPermille, cudaStream_t stream);
// Output dtype != input dtype (f32 <-> f16/bf16): out-of-place on registered buffers.
bool castSupported(DataType in, DataType out);
void launchCastAllreduce(const CommArgs& a, const PeerPtrs& ins, void* mcIn, const PeerPtrs& outs, size_t count,
                         DataType dt, DataType outDt, ReduceOp op, float scale, bool vectorOk, int blocks,
                         cudaStream_t stream);
// Kernel entry points (for occupancy queries: grids must stay co-resident).
const void* twoShotKernelFor(DataType dt, int nranks, int unroll);
const void* nvlsKernelFor(DataType dt, int unroll);
const void* castKernelFor(DataType in, DataType out);

// pipeline_kernels.cu — arbitrary pointers through the pool, 3-stage in-kernel pipeline.
const void* pipelinedKernelFor(DataType dt, bool mc, int nranks);
void launchPipelinedAllreduce(const CommArgs& a, const void* in, void* out, size_t count, DataType dt, ReduceOp op,
                              float scale, const PeerPtrs& stage, void* mcStage, int tileVecs, int exchangeThreads,
                              const LocalPtrs& extra, int blocks, cudaStream_t stream);

// collective_kernels.cu -----------------------------------------------------------------------
void launchBroadcast(const CommArgs& a, const PeerPtrs& bufs, void* mc, size_t bytes, int root, int mode, bool vec,
                     int blocks, int tile, cudaStream_t stream);
void launchGatherPush(const CommArgs& a, const void* in, const PeerPtrs& outs, void* mcOut, const size_t* offs,
                      const size_t* lens, int onlyDst, bool vec, int blocks, cudaStream_t stream, bool tma = false);
void launchAlltoallPush(const CommArgs& a, const void* in, const PeerPtrs& outs, const size_t* sendOff,
                        const size_t* sendLen, const size_t* dstOff, const size_t* recvOffTable, int onlySrc,
                        bool vec, int blocks, cudaStream_t stream);
void launchReducePull(const CommArgs& a, const PeerPtrs& ins, void* mcIn, void* out, const size_t* elemOff,
                      const size_t* elemLen, DataType dt, ReduceOp op, float scale, bool vec, bool useMc, int blocks,
                      cudaStream_t stream);
// The same two collectives with a dtype conversion (one of castSupported's pairs, dt != outDt).
// Offsets and lengths are in elements. reduce_scatter: fp32 accumulation, scale, one rounding
// to outDt, never multicast. allgather: each block converted once, no scale.
void launchReducePullCast(const CommArgs& a, const PeerPtrs& ins, void* out, const size_t* elemOff,
                          const size_t* elemLen, DataType dt, DataType outDt, ReduceOp op, float scale, bool vec,
                          int blocks, cudaStream_t stream);
void launchGatherPushCast(const CommArgs& a, const void* in, const PeerPtrs& outs, const size_t* elemOff,
                          const size_t* elemLen, DataType dt, DataType outDt, bool vec, int blocks,
                          cudaStream_t stream);
// Entry points, for occupancy queries (every CTA of a collective kernel must be resident).
const void* broadcastKernelPtr();
const void* gatherPushKernelPtr();
const void* gatherBulkKernelPtr();
const void* alltoallPushKernelPtr();
const void* reducePullKernelPtr(DataType dt, int nranks);
const void* reducePullCastKernelFor(DataType in, DataType out, int nranks);  // nullptr: unsupported pair
const void* gatherPushCastKernelFor(DataType in, DataType out);
// Flag-in-data exchange for small messages (no barrier): mode 0 = allgather (my block to
// everyone), 1 = alltoall (block j of my input to rank j). `bytes` per block, uniform.
void launchLLExchange(const CommArgs& a, const void* in, void* out, size_t bytes, int mode, const PeerPtrs& ll,
                      size_t srcStride, size_t parityStride, int blocks, int threads, cudaStream_t stream);

// p2p_kernels.cu — point-to-point between two ranks through the receiver's mailbox ring.
// sendBytes == 0 / recvBytes == 0 disables that role; both set = fused send+recv (one launch).
void launchP2p(const CommArgs& a, const void* sendPtr, size_t sendBytes, int dst, void* recvPtr, size_t recvBytes,
               int src, const PeerPtrs& mailbox, size_t boxStride, size_t slotBytes, int nslots, int lanes,
               cudaStream_t stream);
// One-sided copy between my memory and a peer-mapped pointer (put / get), whole grid.
// tma: stream through shared memory with cp.async.bulk (one issuing thread per CTA) when the
// pointers are 16-byte aligned; LDG/STG otherwise.
void launchPeerCopy(void* dst, const void* src, size_t bytes, int blocks, cudaStream_t stream, bool tma = false);
// Zero-copy neighbour exchange: write `sendBytes` straight into `remote` (the peer mapping of
// dst's receive buffer) once dst has signalled ready, and wait for src's data to have landed in
// my own buffer. `blocks` must be the same on both ends of a transfer.
void launchExchange(const CommArgs& a, const void* sendPtr, size_t sendBytes, int dst, void* remote, size_t recvBytes,
                    int src, int blocks, bool tma, cudaStream_t stream);

// reduce_kernels.cu — local element-wise ops: dst = dst (op) src, and
// multi-source reduce / broadcast between buffers visible to one device.
void launchLocalReduce(void* dst, const void* src, size_t count, DataType dt, ReduceOp op, cudaStream_t stream);
void launchLocalReduceMany(void* dst, const void* const* srcs, int nsrc, size_t count, DataType dt, ReduceOp op,
                           cudaStream_t stream);
void launchLocalBroadcast(void* const* dsts, int ndst, const void* src, size_t bytes, cudaStream_t stream);
// Every buffer := scale * reduce(all buffers) in one pass (fused reduce + broadcast).
void launchLocalAllreduceMany(void* const* bufs, int n, size_t count, DataType dt, ReduceOp op, float scale,
                              cudaStream_t stream);
void launchFill(void* dst, size_t count, DataType dt, double start, double stride, cudaStream_t stream);
// Device-side check of buf[i] == start + stride*i; deviceResult = {mismatch count, min(bad index + 1)}
// (initialise to {0, ~0ull}).
void launchVerify(const void* buf, size_t count, DataType dt, double start, double stride, double rtol, double atol,
                  unsigned long long* deviceResult, cudaStream_t stream);
void launchSpin(long long cycles, cudaStream_t stream);
// Launch shape of the single-rank fused step (localAllreduceManyKernel): CTAs per SM, packs per
// thread and trip, contiguous tile per CTA or grid stride. Default from GLB_LOCAL_SHAPE.
void setLocalAllreduceShape(int ctasPerSm, int unroll, bool tiled);

}  // namespace cuda
}  // namespace glb
