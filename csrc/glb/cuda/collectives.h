// Host-side API of the CUDA-buffer collectives: argument checking, variant
// selection per message size and kernel launch. Every call is asynchronous on the
// given stream (a single kernel launch for registered buffers) and must be issued
// in the same order by every rank of the PeerContext.
//
// Buffers come in two flavours:
//   * PeerBuffer (registerBuffer / allocSymmetric): zero-copy, kernels read and
//     write the peers' copies directly;
//   * arbitrary device pointers: staged through the symmetric pool.
#pragma once

#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "glb/cuda/peer_context.h"
#include "glb/cuda/tuning.h"
#include "glb/types.h"

namespace glb {
namespace cuda {

enum class AllreduceAlgo : int {
  AUTO = 0,
  ONE_SHOT = 1,
  TWO_SHOT = 2,
  NVLS = 3,
  LL = 4,         // flag-in-data one-shot, no barrier (smallest messages)
  PIPELINED = 5,  // arbitrary pointers: in-kernel copy-in / exchange / copy-out pipeline through the pool
  HYBRID = 6,     // NVLS on one part of the vector + peer-to-peer two-shot on the rest, concurrently
  // Literal schedules of the reference's named algorithms, executed by the
  // step-table kernel over peer pointers (schedule_kernels.cu).
  RING = 10,
  RING_CHUNKED = 11,
  HALVING_DOUBLING = 12,
  BCUBE = 13,
  HALVING_DOUBLING_PIPELINED = 14,
};

const char* allreduceAlgoName(AllreduceAlgo a);

AllreduceAlgo allreduceAlgoFromName(const std::string& name);

// Process-wide knobs (initialised from GLB_CUDA_* env vars). Per-size decisions come from
// the measured tuning table (tuning.h); these are the fallbacks and global caps.
struct Tuning {
  size_t llMaxBytes = 16 * 1024;        // flag-in-data one-shot while bytes <= this
  size_t oneShotMaxBytes = 256 * 1024;  // barrier one-shot while bytes <= this / P; above: two-shot / NVLS
  size_t nvlsMinBytes = 32 * 1024;      // >= : NVLS when the buffer has a multicast alias (and P > 2)
  int maxBlocks = 128;                  // CTAs for the bandwidth kernels (clamped to the co-residency cap)
  int oneShotBlocks = 8;
  bool nvlsReduceScatter = false;       // multimem.ld_reduce in reduce_scatter / reduce: measured slower than the
                                        // P2P pull at P=4 (403 vs 343 us @256 MB) and equal at P=8, so off by default
  int copyBlocks = 296;                 // CTAs for the store-only kernels (40 regs: 2-3 CTAs per SM)
  int alltoallvBlocks = 64;             // fixed grid of the v-variant (sizes are rank-local, the grid must not be)
  size_t bcastDirectMaxBytes = 256 * 1024;  // <= : root pushes everything itself
  size_t bcastRelayMinBytes = 64u << 20;    // >= : chunk-pipelined relay broadcast (P > 2; measured cross-over 32-256 MB)
  int pipeTile = 1024;                  // 16-byte groups per tile of the pipelined kernel (power of two)
  int pipeExchangeThreads = 256;        // threads of each CTA that drive NVLink in the pipelined kernel
  bool tmaCopies = false;               // put / get / large allgather through cp.async.bulk (TMA) instead of LDG/STG
                                        // when no table entry decides (GLB_CUDA_TMA)
};
Tuning& tuning();
// Number of collective kernels launched by this process so far.
uint64_t launchCount();
void noteLaunch(unsigned n = 1);  // local (non-collective) kernels report here

// What AUTO resolves to for a call, with the launch shape from the tuning table.
struct AllreducePlan {
  AllreduceAlgo algo = AllreduceAlgo::AUTO;
  LaunchCfg cfg;
  int tile = 0;
  bool fromTable = false;
};
AllreducePlan planAllreduce(PeerContext& pc, size_t bytes, DataType dt, ReduceOp op, BufKind kind);
// Which variant AUTO resolves to for this call (legacy signature).
AllreduceAlgo chooseAllreduce(PeerContext& pc, size_t bytes, DataType dt, ReduceOp op, bool registered,
                              bool hasMulticast);

// Optional per-call arguments of allreduce / reduce_scatter / reduce: the fused epilogue.
struct Epilogue {
  double scale = 1.0;           // multiply the reduced value before the final rounding (AVG: 1 / P)
  bool castOutput = false;      // store as `outDtype` instead of the input dtype
  DataType outDtype = DataType::FLOAT32;
  LocalPtrs extra;              // more local inputs (same count / dtype): folded in, and overwritten with the result
  // Pin the launch shape (tuner / sweeps); 0 = from the tuning table.
  int blocks = 0;
  int unroll = 0;
  int tile = 0;
};

void barrier(PeerContext& pc, cudaStream_t stream);

// In place on a registered / symmetric buffer (count elements from byteOffset).
void allreduce(PeerContext& pc, const PeerBuffer& buf, size_t byteOffset, size_t count, DataType dt, ReduceOp op,
               AllreduceAlgo algo, cudaStream_t stream, const Epilogue& ep = Epilogue());

// Arbitrary device pointers (in may equal out): LL / one-shot for small messages, the
// pipelined kernel above. With ep.castOutput `out` holds ep.outDtype elements (small
// messages only; larger ones need registered buffers, see allreduceCast).
void allreduce(PeerContext& pc, const void* in, void* out, size_t count, DataType dt, ReduceOp op,
               AllreduceAlgo algo, cudaStream_t stream, const Epilogue& ep = Epilogue());

// Out of place between two registered buffers with different dtypes (f32 <-> f16 / bf16):
// fp32 accumulation, one rounding to `outDt`.
void allreduceCast(PeerContext& pc, const PeerBuffer& in, size_t inOffset, const PeerBuffer& out, size_t outOffset,
                   size_t count, DataType dt, DataType outDt, ReduceOp op, cudaStream_t stream,
                   const Epilogue& ep = Epilogue());


// ---- data movement -------------------------------------------------------------------
// `buf`/`out` arguments are registered or symmetric buffers; plain-pointer
// overloads stage through the pool (payload limited to the pool's bulk region).

// In place: root's bytes replace everyone's.
void broadcast(PeerContext& pc, const PeerBuffer& buf, size_t byteOffset, size_t bytes, int root,
               cudaStream_t stream);
void broadcast(PeerContext& pc, void* ptr, size_t bytes, int root, cudaStream_t stream);

// Rank r's `in` (bytesPerRank[r] bytes) lands at the prefix-sum offset in every out.
void allgatherv(PeerContext& pc, const void* in, const PeerBuffer& out, size_t outOffset,
                const std::vector<size_t>& bytesPerRank, cudaStream_t stream);
void allgatherv(PeerContext& pc, const void* in, void* out, const std::vector<size_t>& bytesPerRank,
                cudaStream_t stream);
// allgatherv with a dtype conversion (f32 -> f16 / bf16 rounds to nearest even, f16 / bf16 ->
// f32 is exact): rank r's `in` (counts[r] ELEMENTS of inDt) lands, converted to outDt, at the
// prefix-sum element offset of every out. Each block is read and converted once. Same dtypes:
// allgatherv.
void allgathervCast(PeerContext& pc, const void* in, DataType inDt, const PeerBuffer& out, size_t outOffset,
                    const std::vector<size_t>& counts, DataType outDt, cudaStream_t stream);
void allgathervCast(PeerContext& pc, const void* in, DataType inDt, void* out, const std::vector<size_t>& counts,
                    DataType outDt, cudaStream_t stream);
// Only `root` receives.
void gatherv(PeerContext& pc, const void* in, const PeerBuffer& out, size_t outOffset,
             const std::vector<size_t>& bytesPerRank, int root, cudaStream_t stream);
void gatherv(PeerContext& pc, const void* in, void* out, const std::vector<size_t>& bytesPerRank, int root,
             cudaStream_t stream);

// Chunk j of my input (sendBytes[j] at the prefix-sum offset) goes to rank j, which
// stores what it gets from rank i at the prefix-sum offset of ITS recvBytes[i].
void alltoallv(PeerContext& pc, const void* in, const std::vector<size_t>& sendBytes, const PeerBuffer& out,
               size_t outOffset, const std::vector<size_t>& recvBytes, cudaStream_t stream);
void alltoallv(PeerContext& pc, const void* in, const std::vector<size_t>& sendBytes, void* out,
               const std::vector<size_t>& recvBytes, cudaStream_t stream);
// Fixed-size alltoall: every chunk is `bytes` long on every rank (this is known to all
// ranks, so the small-message LL kernel and size-dependent grids are safe here).
void alltoall(PeerContext& pc, const void* in, const PeerBuffer& out, size_t outOffset, size_t bytes,
              cudaStream_t stream);
void alltoall(PeerContext& pc, const void* in, void* out, size_t bytes, cudaStream_t stream);
// Root's input holds P chunks of `bytes`; chunk j lands in rank j's out.
void scatter(PeerContext& pc, const void* in, const PeerBuffer& out, size_t outOffset, size_t bytes, int root,
             cudaStream_t stream);
void scatter(PeerContext& pc, const void* in, void* out, size_t bytes, int root, cudaStream_t stream);

// Rank r gets elements [prefix(counts, r), +counts[r]) of the reduction in `out`.
void reduce_scatter(PeerContext& pc, const PeerBuffer& in, size_t inOffset, void* out,
                    const std::vector<size_t>& counts, DataType dt, ReduceOp op, cudaStream_t stream,
                    double scale = 1.0);
void reduce_scatter(PeerContext& pc, const void* in, void* out, const std::vector<size_t>& counts, DataType dt,
                    ReduceOp op, cudaStream_t stream, double scale = 1.0);
// reduce_scatter of `dt` inputs into an `outDt` output (f32 <-> f16 / bf16): fp32 accumulation,
// `scale` on the accumulator, one rounding to outDt. One barrier kernel at every size (no LL
// variant) and never multicast. Same dtypes: reduce_scatter.
void reduceScatterCast(PeerContext& pc, const PeerBuffer& in, size_t inOffset, void* out,
                       const std::vector<size_t>& counts, DataType dt, DataType outDt, ReduceOp op,
                       cudaStream_t stream, double scale = 1.0);
void reduceScatterCast(PeerContext& pc, const void* in, void* out, const std::vector<size_t>& counts, DataType dt,
                       DataType outDt, ReduceOp op, cudaStream_t stream, double scale = 1.0);
// Reduction of every rank's `in` delivered to root's `out` (both registered).
void reduce(PeerContext& pc, const PeerBuffer& in, size_t inOffset, const PeerBuffer& out, size_t outOffset,
            size_t count, DataType dt, ReduceOp op, int root, cudaStream_t stream);
void reduce(PeerContext& pc, const void* in, void* out, size_t count, DataType dt, ReduceOp op, int root,
            cudaStream_t stream);

// ---- point to point ----------------------------------------------------------------------------
// Device buffers between two ranks over NVLink (p2p_kernels.cu). Sends and receives between
// a pair of ranks match in posting order. sendrecv posts both directions in ONE kernel, the
// right call for ring / pipeline exchanges (a separate send and recv on one stream would
// serialise and, for messages larger than the mailbox ring, wait for each other).
void send(PeerContext& pc, const void* ptr, size_t bytes, int dst, cudaStream_t stream);
void recv(PeerContext& pc, void* ptr, size_t bytes, int src, cudaStream_t stream);
void sendrecv(PeerContext& pc, const void* sendPtr, size_t sendBytes, int dst, void* recvPtr, size_t recvBytes,
              int src, cudaStream_t stream);
// One-sided on registered memory: my [local, local+bytes) <-> rank `peer`'s copy of `remote`
// at remoteOffset. Completion is stream order on the initiator; the target learns about it
// through a later collective / barrier / message (RDMA semantics, as
// gloo/transport/unbound_buffer.h:128-152).
// Zero-copy sendrecv for a peer-mapped receive buffer that every rank uses at the same offset
// (ring attention's K/V double buffer, a pipeline stage's activation slot): my `sendBytes` are
// written straight into recvBuf on `dst` at recvOffset, `src` writes into mine. One kernel, one
// pass over the data, one flag round trip per call. After it completes on `stream`, my
// recvBuf[recvOffset, +recvBytes) holds src's payload; my sendPtr may be reused. The receive
// range must not be read or written by work queued behind the PREVIOUS exchange's consumer
// until this call is enqueued (the kernel start is the "ready to be overwritten" signal).
void exchange(PeerContext& pc, const void* sendPtr, size_t sendBytes, int dst, const PeerBuffer& recvBuf,
              size_t recvOffset, size_t recvBytes, int src, cudaStream_t stream);
void put(PeerContext& pc, const void* local, const PeerBuffer& remote, size_t remoteOffset, size_t bytes, int peer,
         cudaStream_t stream);
void get(PeerContext& pc, void* local, const PeerBuffer& remote, size_t remoteOffset, size_t bytes, int peer,
         cudaStream_t stream);

}  // namespace cuda
}  // namespace glb
