#include "glb/cuda/collectives.h"

#include <algorithm>
#include <atomic>

#include "glb/common/utils.h"
#include "glb/cuda/kernels.h"
#include "glb/cuda/trace.h"

namespace glb {
namespace cuda {

const char* allreduceAlgoName(AllreduceAlgo a) {
  switch (a) {
    case AllreduceAlgo::AUTO: return "auto";
    case AllreduceAlgo::ONE_SHOT: return "one_shot";
    case AllreduceAlgo::TWO_SHOT: return "two_shot";
    case AllreduceAlgo::NVLS: return "nvls";
    case AllreduceAlgo::LL: return "ll";
    case AllreduceAlgo::PIPELINED: return "pipelined";
    case AllreduceAlgo::HYBRID: return "hybrid";
    case AllreduceAlgo::RING: return "ring";
    case AllreduceAlgo::RING_CHUNKED: return "ring_chunked";
    case AllreduceAlgo::HALVING_DOUBLING: return "halving_doubling";
    case AllreduceAlgo::BCUBE: return "bcube";
    case AllreduceAlgo::HALVING_DOUBLING_PIPELINED: return "halving_doubling_pipelined";
  }
  return "?";
}

AllreduceAlgo allreduceAlgoFromName(const std::string& n) {
  for (AllreduceAlgo a : {AllreduceAlgo::AUTO, AllreduceAlgo::ONE_SHOT, AllreduceAlgo::TWO_SHOT, AllreduceAlgo::NVLS,
                          AllreduceAlgo::LL, AllreduceAlgo::PIPELINED, AllreduceAlgo::HYBRID, AllreduceAlgo::RING,
                          AllreduceAlgo::RING_CHUNKED,
                          AllreduceAlgo::HALVING_DOUBLING, AllreduceAlgo::BCUBE,
                          AllreduceAlgo::HALVING_DOUBLING_PIPELINED}) {
    if (n == allreduceAlgoName(a)) return a;
  }
  return AllreduceAlgo::AUTO;
}

Tuning& tuning() {
  static Tuning t = [] {
    Tuning x;
    x.llMaxBytes = static_cast<size_t>(envInt("CUDA_LL_MAX", static_cast<long>(x.llMaxBytes)));
    x.oneShotMaxBytes = static_cast<size_t>(envInt("CUDA_ONESHOT_MAX", static_cast<long>(x.oneShotMaxBytes)));
    x.nvlsMinBytes = static_cast<size_t>(envInt("CUDA_NVLS_MIN", static_cast<long>(x.nvlsMinBytes)));
    x.maxBlocks = static_cast<int>(envInt("CUDA_BLOCKS", x.maxBlocks));
    x.oneShotBlocks = static_cast<int>(envInt("CUDA_ONESHOT_BLOCKS", x.oneShotBlocks));
    x.copyBlocks = static_cast<int>(envInt("CUDA_COPY_BLOCKS", x.copyBlocks));
    x.alltoallvBlocks = static_cast<int>(envInt("CUDA_ALLTOALLV_BLOCKS", x.alltoallvBlocks));
    x.nvlsReduceScatter = envFlag("CUDA_NVLS_REDUCE_SCATTER", x.nvlsReduceScatter);
    setOneShotPush(envFlag("CUDA_ONESHOT_PUSH", true));
    x.bcastDirectMaxBytes = static_cast<size_t>(envInt("CUDA_BCAST_DIRECT_MAX", static_cast<long>(x.bcastDirectMaxBytes)));
    x.bcastRelayMinBytes = static_cast<size_t>(envInt("CUDA_BCAST_RELAY_MIN", static_cast<long>(x.bcastRelayMinBytes)));
    x.pipeTile = static_cast<int>(envInt("CUDA_PIPE_TILE", x.pipeTile));
    x.pipeExchangeThreads = static_cast<int>(envInt("CUDA_PIPE_XTHREADS", x.pipeExchangeThreads));
    x.tmaCopies = envFlag("CUDA_TMA", x.tmaCopies);
    return x;
  }();
  return t;
}

namespace {

// Layout of the staging area: two one-shot halves, then the bulk region.
struct StageLayout {
  size_t half;       // bytes of one one-shot half
  size_t bulkOff;    // start of the bulk (pipelined / staged collectives) region
  size_t bulkBytes;
};

StageLayout layoutOf(const PeerContext& pc) {
  StageLayout l;
  l.half = std::min<size_t>(roundUp(std::max<size_t>(tuning().oneShotMaxBytes, 4096), 4096), pc.stageBytes() / 4);
  l.bulkOff = 2 * l.half;
  l.bulkBytes = pc.stageBytes() - l.bulkOff;
  return l;
}

int blocksFor(const PeerContext& pc, size_t vecsPerRank, int unrollHint, int cap) {
  size_t want = ceilDiv(std::max<size_t>(vecsPerRank, 1), static_cast<size_t>(kThreads) * unrollHint);
  int b = static_cast<int>(std::min<size_t>(want, static_cast<size_t>(cap)));
  return std::max(1, std::min(b, pc.maxBlocks()));
}

std::atomic<uint64_t> gLaunches{0};

void checkLaunch(const char* what) {
  gLaunches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) GLB_THROW(Exception, what, ": kernel launch failed: ", cudaGetErrorString(e));
}

// Everything a collective does before it launches: device, health, stream order, and the
// host rendezvous needed when ranks share a GPU.
void prologue(PeerContext& pc, cudaStream_t stream) {
  pc.checkHealth();
  pc.orderStreams(stream);
  pc.launchGuard();
}

// ... and after it has launched.
void finish(PeerContext& pc, cudaStream_t stream, const char* what) {
  checkLaunch(what);
  pc.markLaunched(stream);
}

float scaleOf(const Epilogue& ep, DataType dt) {
  if (ep.scale == 1.0) return 1.0f;
  GLB_ENFORCE(dt == DataType::FLOAT32 || dt == DataType::FLOAT64 || dt == DataType::FLOAT16 || dt == DataType::BFLOAT16,
              "a scale epilogue needs a floating-point buffer");
  return static_cast<float>(ep.scale);
}

// Grid of a bandwidth kernel: enough CTAs for the work, never more than the table / knob
// says, never more than can be co-resident.
int clampBlocks(PeerContext& pc, const void* kernel, int wanted, size_t vecsPerRank, int unroll) {
  const size_t need = ceilDiv(std::max<size_t>(vecsPerRank, 1), static_cast<size_t>(kThreads) * std::max(unroll, 1));
  int b = static_cast<int>(std::min<size_t>(need, static_cast<size_t>(std::max(wanted, 1))));
  return std::max(1, std::min(b, pc.coResidentBlocks(kernel)));
}

int defaultUnroll(AllreduceAlgo a, int P) {
  if (a == AllreduceAlgo::NVLS) return 4;
  return P == 2 ? 4 : 2;
}

}  // namespace

uint64_t launchCount() { return gLaunches.load(); }
void noteLaunch(unsigned n) { gLaunches.fetch_add(n, std::memory_order_relaxed); }

AllreducePlan planAllreduce(PeerContext& pc, size_t bytes, DataType dt, ReduceOp op, BufKind kind) {
  const auto& t = tuning();
  const int P = std::max(pc.size, 1);
  const auto l = layoutOf(pc);
  AllreducePlan plan;
  auto usable = [&](AllreduceAlgo a) {
    switch (a) {
      case AllreduceAlgo::LL: return bytes <= pc.llMaxBytes();
      case AllreduceAlgo::ONE_SHOT: return roundUp(bytes, 16) <= l.half;
      case AllreduceAlgo::NVLS: return kind == BufKind::SYMMETRIC && nvlsSupports(dt, op);
      case AllreduceAlgo::HYBRID:
        return kind == BufKind::SYMMETRIC && nvlsSupports(dt, op) && hybridKernelFor(dt, pc.size) != nullptr;
      case AllreduceAlgo::TWO_SHOT: return kind != BufKind::USER;
      case AllreduceAlgo::PIPELINED: return kind == BufKind::USER;
      default: return false;
    }
  };
  if (const TuneEntry* e = TuningTable::get().lookup("allreduce", P, kind, bytes)) {
    AllreduceAlgo a = allreduceAlgoFromName(e->algo);
    if (a != AllreduceAlgo::AUTO && usable(a)) {
      plan.algo = a;
      plan.cfg.blocks = e->blocks;
      plan.cfg.unroll = e->unroll;
      plan.tile = e->tile;
      plan.fromTable = true;
      return plan;
    }
  }
  // Built-in fallback. One-shot moves (P-1)*S into every GPU, so its break-even shrinks
  // with P; in-switch reduction moves ~S(1+1/P) per direction against 2S(P-1)/P for
  // two-shot: a win from P = 4 up, a loss at P = 2.
  if (bytes <= t.llMaxBytes && usable(AllreduceAlgo::LL)) {
    plan.algo = AllreduceAlgo::LL;
  } else if (bytes <= t.oneShotMaxBytes / static_cast<size_t>(P) && usable(AllreduceAlgo::ONE_SHOT)) {
    plan.algo = AllreduceAlgo::ONE_SHOT;
  } else if (kind == BufKind::USER) {
    plan.algo = AllreduceAlgo::PIPELINED;
  } else if (P > 2 && bytes >= t.nvlsMinBytes && usable(AllreduceAlgo::NVLS)) {
    plan.algo = AllreduceAlgo::NVLS;
  } else {
    plan.algo = AllreduceAlgo::TWO_SHOT;
  }
  plan.cfg.blocks = 0;
  plan.cfg.unroll = 0;
  return plan;
}

AllreduceAlgo chooseAllreduce(PeerContext& pc, size_t bytes, DataType dt, ReduceOp op, bool registered,
                              bool hasMulticast) {
  const BufKind kind = !registered ? BufKind::USER : (hasMulticast ? BufKind::SYMMETRIC : BufKind::REGISTERED);
  return planAllreduce(pc, bytes, dt, op, kind).algo;
}

void barrier(PeerContext& pc, cudaStream_t stream) {
  GLB_TRACE_RANGE("glb::cuda::barrier");
  DeviceGuard g(pc.device);
  prologue(pc, stream);
  launchBarrier(pc.comm(), stream);
  finish(pc, stream, "barrier");
}

namespace {

void runLL(PeerContext& pc, const void* in, void* out, size_t count, DataType dt, DataType outDt, ReduceOp op,
           float scale, const LocalPtrs& extra, int blocksHint, cudaStream_t stream) {
  const size_t es = elementSize(dt);
  GLB_ENFORCE_LE(count * es, pc.llMaxBytes(), "LL allreduce limited to ", pc.llMaxBytes(), " bytes");
  const size_t units = ceilDiv(count * es, size_t(8));
  int threads = static_cast<int>(std::min<size_t>(kThreads, roundUp(std::max<size_t>(units, 32), 32)));
  int blocks = static_cast<int>(ceilDiv(units, static_cast<size_t>(threads)));
  blocks = std::max(1, std::min({blocks, blocksHint > 0 ? blocksHint : 16, pc.maxBlocks()}));  // no barrier: no co-residency need
  launchLLAllreduce(pc.comm(), in, out, count, dt, outDt, op, scale, pc.llPtrs(), pc.llSrcStride(), pc.llParityStride(),
                    extra, blocks, threads, stream);
}

// Single rank with a dtype conversion: the LL kernel degenerates to a local scale and
// convert; it runs in pieces the LL region accepts.
void localCast(PeerContext& pc, const void* in, void* out, size_t count, DataType dt, DataType outDt, ReduceOp op,
               float scale, cudaStream_t stream, const char* what) {
  const size_t piece = pc.llMaxBytes() / elementSize(dt);
  pc.checkHealth();
  for (size_t done = 0; done < count; done += piece) {
    const size_t n = std::min(piece, count - done);
    runLL(pc, static_cast<const char*>(in) + done * elementSize(dt), static_cast<char*>(out) + done * elementSize(outDt),
          n, dt, outDt, op, scale, LocalPtrs(), 0, stream);
    checkLaunch(what);
  }
}

void runOneShot(PeerContext& pc, const void* in, void* out, size_t count, DataType dt, ReduceOp op, float scale,
                const LocalPtrs& extra, int blocksHint, cudaStream_t stream) {
  const auto l = layoutOf(pc);
  const size_t bytes = count * elementSize(dt);
  GLB_ENFORCE_LE(roundUp(bytes, 16), l.half, "one-shot allreduce limited to ", l.half, " bytes");
  const int blocks = blocksFor(pc, ceilDiv(bytes, size_t(16)), 1, blocksHint > 0 ? blocksHint : tuning().oneShotBlocks);
  launchOneShotAllreduce(pc.comm(), in, out, count, dt, op, scale, pc.stagePtrs(0), l.half, extra, blocks, stream);
}

void runPipelined(PeerContext& pc, const void* in, void* out, size_t count, DataType dt, ReduceOp op, float scale,
                  const LocalPtrs& extra, const AllreducePlan& plan, cudaStream_t stream) {
  const auto l = layoutOf(pc);
  const size_t es = elementSize(dt);
  const size_t groups = ceilDiv(count * es, size_t(16));
  const bool mc = pc.nvlsAvailable() && pc.size > 2 && nvlsSupports(dt, op);
  const void* kernel = pipelinedKernelFor(dt, mc, pc.size);
  int blocks = plan.cfg.blocks > 0 ? plan.cfg.blocks : tuning().maxBlocks;
  blocks = std::max(1, std::min(blocks, pc.coResidentBlocks(kernel)));
  // Tile: a power of two, small enough for three slots in the bulk region and for a few
  // steps of pipelining on mid-sized messages.
  int tile = plan.tile > 0 ? plan.tile : tuning().pipeTile;
  auto chunkBytes = [&](int tl, int bl) { return static_cast<size_t>(pc.size) * bl * tl * 16; };
  int t2 = 16;
  while (t2 * 2 <= tile) t2 *= 2;
  tile = t2;
  while (tile > 16 && (3 * chunkBytes(tile, blocks) > l.bulkBytes || groups * 16 < 4 * chunkBytes(tile, blocks))) tile /= 2;
  while (blocks > 1 && groups * 16 < chunkBytes(tile, blocks)) blocks = (blocks + 1) / 2;  // tiny messages: fewer CTAs
  GLB_ENFORCE_LE(3 * chunkBytes(tile, blocks), l.bulkBytes, "staging pool too small for the pipelined allreduce; raise GLB_CUDA_STAGE_MB");
  // cfg.unroll doubles as "exchange warps" for this kernel (0 = the pipeExchangeThreads knob).
  int xthreads = plan.cfg.unroll > 0 ? plan.cfg.unroll * 32 : tuning().pipeExchangeThreads;
  xthreads = std::max(32, std::min(kThreads - 32, xthreads / 32 * 32));
  launchPipelinedAllreduce(pc.comm(), in, out, count, dt, op, scale, pc.stagePtrs(l.bulkOff),
                           mc ? pc.stageMc(l.bulkOff) : nullptr, tile, xthreads, extra, blocks, stream);
}

}  // namespace

void allreduce(PeerContext& pc, const PeerBuffer& buf, size_t byteOffset, size_t count, DataType dt, ReduceOp op,
               AllreduceAlgo algo, cudaStream_t stream, const Epilogue& ep) {
  GLB_TRACE_RANGE("glb::cuda::allreduce");
  pc.checkHealth();
  if (count == 0) return;
  const size_t es = elementSize(dt);
  const size_t bytes = count * es;
  GLB_ENFORCE_LE(byteOffset + bytes, buf.bytes, "allreduce range exceeds the registered buffer");
  GLB_ENFORCE(op != ReduceOp::CUSTOM, "custom reductions run on the host path only");
  GLB_ENFORCE(!ep.castOutput || ep.outDtype == dt, "in-place allreduce cannot change the dtype; use allreduceCast");
  const float scale = scaleOf(ep, dt);
  DeviceGuard g(pc.device);
  char* local = static_cast<char*>(buf.local) + byteOffset;
  // Single rank: the buffer already holds the result unless there is something to fold or
  // scale. GLB_CUDA_FORCE_KERNELS=1 still launches the collective kernel (loopback on local
  // memory) so it can be profiled with Nsight Compute.
  if (pc.size == 1 && !envFlag("CUDA_FORCE_KERNELS", false)) {
    if (ep.extra.n > 0 || scale != 1.0f) {
      std::vector<void*> all{local};
      for (int k = 0; k < ep.extra.n; k++) all.push_back(ep.extra.p[k]);
      launchLocalAllreduceMany(all.data(), static_cast<int>(all.size()), count, dt, op, scale, stream);
      checkLaunch("allreduce(local)");
    }
    return;
  }
  const bool hasMc = buf.mc != nullptr && byteOffset % 16 == 0;
  const BufKind kind = hasMc ? BufKind::SYMMETRIC : BufKind::REGISTERED;
  AllreducePlan plan;
  if (algo == AllreduceAlgo::AUTO) {
    plan = planAllreduce(pc, bytes, dt, op, kind);
    algo = plan.algo;
    if (algo == AllreduceAlgo::HYBRID && ep.extra.n > 0) {  // the hybrid kernel takes one pointer
      algo = AllreduceAlgo::NVLS;
      plan.cfg = LaunchCfg();
    }
  }
  if (ep.blocks > 0) plan.cfg.blocks = ep.blocks;
  if (ep.unroll > 0) plan.cfg.unroll = ep.unroll;
  prologue(pc, stream);
  switch (algo) {
    case AllreduceAlgo::LL:
      runLL(pc, local, local, count, dt, dt, op, scale, ep.extra, plan.cfg.blocks, stream);
      break;
    case AllreduceAlgo::ONE_SHOT:
      runOneShot(pc, local, local, count, dt, op, scale, ep.extra, plan.cfg.blocks, stream);
      break;
    case AllreduceAlgo::NVLS: {
      GLB_ENFORCE(hasMc, "NVLS allreduce needs a multicast-bound (symmetric) buffer");
      GLB_ENFORCE(nvlsSupports(dt, op), "NVLS supports sum over float32/float16/bfloat16 only");
      LaunchCfg cfg = plan.cfg;
      if (cfg.unroll == 0) cfg.unroll = defaultUnroll(algo, pc.size);
      cfg.blocks = clampBlocks(pc, nvlsKernelFor(dt, cfg.unroll), cfg.blocks > 0 ? cfg.blocks : tuning().maxBlocks,
                               ceilDiv(bytes, size_t(16)) / pc.size, cfg.unroll);
      launchNvlsAllreduce(pc.comm(), static_cast<char*>(buf.mc) + byteOffset, buf.ptrsAt(byteOffset), count, dt, scale,
                          ep.extra, cfg, stream);
      break;
    }
    case AllreduceAlgo::HYBRID: {
      GLB_ENFORCE(hasMc && nvlsSupports(dt, op) && hybridKernelFor(dt, pc.size) != nullptr && ep.extra.n == 0,
                  "hybrid allreduce: sum of f32/f16/bf16 on a multicast-bound buffer, 4 or 8 ranks, one pointer");
      // cfg.blocks = all CTAs, cfg.unroll = CTAs of the NVLS part, tile = per-mille of the vector done peer to peer
      int blocks = plan.cfg.blocks > 0 ? plan.cfg.blocks : 148;
      blocks = std::max(2, std::min(blocks, pc.coResidentBlocks(hybridKernelFor(dt, pc.size))));
      const int nvlsBlocks = std::max(1, std::min(plan.cfg.unroll > 0 ? plan.cfg.unroll : 32, blocks - 1));
      const int permille = std::max(0, std::min((ep.tile > 0 ? ep.tile : plan.tile > 0 ? plan.tile : 175), 900));
      launchHybridAllreduce(pc.comm(), static_cast<char*>(buf.mc) + byteOffset, buf.ptrsAt(byteOffset), count, dt, scale,
                            blocks, nvlsBlocks, static_cast<unsigned>(permille), stream);
      break;
    }
    case AllreduceAlgo::TWO_SHOT: {
      const bool vectorOk = buf.vectorOk && byteOffset % 16 == 0;
      LaunchCfg cfg = plan.cfg;
      if (cfg.unroll == 0) cfg.unroll = defaultUnroll(algo, pc.size);
      cfg.blocks = clampBlocks(pc, twoShotKernelFor(dt, pc.size, cfg.unroll), cfg.blocks > 0 ? cfg.blocks : tuning().maxBlocks,
                               bytes / 16 / pc.size, cfg.unroll);
      launchTwoShotAllreduce(pc.comm(), buf.ptrsAt(byteOffset), count, dt, op, scale, vectorOk, ep.extra, cfg, stream);
      break;
    }
    case AllreduceAlgo::PIPELINED:
      plan.tile = ep.tile > 0 ? ep.tile : plan.tile;
      runPipelined(pc, local, local, count, dt, op, scale, ep.extra, plan, stream);
      break;
    default:
      GLB_THROW_INVALID_OPERATION_EXCEPTION("allreduce: algorithm ", allreduceAlgoName(algo),
                                            " is not available on this entry point");
  }
  finish(pc, stream, "allreduce");
}

void allreduce(PeerContext& pc, const void* in, void* out, size_t count, DataType dt, ReduceOp op,
               AllreduceAlgo algo, cudaStream_t stream, const Epilogue& ep) {
  GLB_TRACE_RANGE("glb::cuda::allreduce(user pointers)");
  pc.checkHealth();
  if (count == 0) return;
  GLB_ENFORCE(op != ReduceOp::CUSTOM, "custom reductions run on the host path only");
  DeviceGuard g(pc.device);
  const size_t es = elementSize(dt);
  const size_t bytes = count * es;
  const DataType outDt = ep.castOutput ? ep.outDtype : dt;
  GLB_ENFORCE(castSupported(dt, outDt), "allreduce: unsupported dtype conversion in the epilogue");
  const float scale = scaleOf(ep, dt);
  if (pc.size == 1 && !envFlag("CUDA_FORCE_KERNELS", false)) {
    if (outDt != dt) {
      // Single rank with a cast: the LL kernel degenerates to a fused fold / scale / convert.
      GLB_ENFORCE_LE(bytes, pc.llMaxBytes(), "allreduce with a dtype conversion on plain pointers is limited to ",
                     pc.llMaxBytes(), " bytes; register the buffers (allreduceCast)");
      pc.checkHealth();
      runLL(pc, in, out, count, dt, outDt, op, scale, ep.extra, 0, stream);
      checkLaunch("allreduce(ll)");
      return;
    }
    if (ep.extra.n > 0 || scale != 1.0f) {
      if (in != out) GLB_CUDA_CHECK(cudaMemcpyAsync(out, in, bytes, cudaMemcpyDeviceToDevice, stream));
      std::vector<void*> all{out};
      for (int k = 0; k < ep.extra.n; k++) all.push_back(ep.extra.p[k]);
      launchLocalAllreduceMany(all.data(), static_cast<int>(all.size()), count, dt, op, scale, stream);
      checkLaunch("allreduce(local)");
    } else if (in != out) {
      GLB_CUDA_CHECK(cudaMemcpyAsync(out, in, bytes, cudaMemcpyDeviceToDevice, stream));
    }
    return;
  }
  AllreducePlan plan;
  if (algo == AllreduceAlgo::AUTO) {
    plan = planAllreduce(pc, bytes, dt, op, BufKind::USER);
    algo = plan.algo;
  }
  if (ep.blocks > 0) plan.cfg.blocks = ep.blocks;
  if (ep.unroll > 0) plan.cfg.unroll = ep.unroll;
  if (ep.tile > 0) plan.tile = ep.tile;
  if (outDt != dt) {
    GLB_ENFORCE_LE(bytes, pc.llMaxBytes(), "allreduce with a dtype conversion on plain pointers is limited to ",
                   pc.llMaxBytes(), " bytes; register the buffers (allreduceCast)");
    algo = AllreduceAlgo::LL;
  }
  // Variants that need peer-visible user memory fall back to the pool path.
  if (algo == AllreduceAlgo::TWO_SHOT || algo == AllreduceAlgo::NVLS) algo = AllreduceAlgo::PIPELINED;
  if (algo == AllreduceAlgo::ONE_SHOT && roundUp(bytes, 16) > layoutOf(pc).half) algo = AllreduceAlgo::PIPELINED;
  if (algo == AllreduceAlgo::LL && bytes > pc.llMaxBytes()) algo = AllreduceAlgo::PIPELINED;
  prologue(pc, stream);
  switch (algo) {
    case AllreduceAlgo::LL: runLL(pc, in, out, count, dt, outDt, op, scale, ep.extra, plan.cfg.blocks, stream); break;
    case AllreduceAlgo::ONE_SHOT: runOneShot(pc, in, out, count, dt, op, scale, ep.extra, plan.cfg.blocks, stream); break;
    case AllreduceAlgo::PIPELINED: runPipelined(pc, in, out, count, dt, op, scale, ep.extra, plan, stream); break;
    default:
      GLB_THROW_INVALID_OPERATION_EXCEPTION("allreduce: algorithm ", allreduceAlgoName(algo), " needs registered buffers");
  }
  finish(pc, stream, "allreduce(user pointers)");
}

void allreduceCast(PeerContext& pc, const PeerBuffer& in, size_t inOffset, const PeerBuffer& out, size_t outOffset,
                   size_t count, DataType dt, DataType outDt, ReduceOp op, cudaStream_t stream, const Epilogue& ep) {
  GLB_TRACE_RANGE("glb::cuda::allreduceCast");
  if (count == 0) return;
  GLB_ENFORCE(dt != outDt && castSupported(dt, outDt), "allreduceCast: supported conversions are f32 <-> f16 / bf16");
  GLB_ENFORCE(op != ReduceOp::CUSTOM, "custom reductions run on the host path only");
  GLB_ENFORCE_LE(inOffset + count * elementSize(dt), in.bytes, "allreduceCast input range exceeds the buffer");
  GLB_ENFORCE_LE(outOffset + count * elementSize(outDt), out.bytes, "allreduceCast output range exceeds the buffer");
  GLB_ENFORCE(ep.extra.n == 0, "allreduceCast takes one input per rank");
  const float scale = scaleOf(ep, DataType::FLOAT32);
  DeviceGuard g(pc.device);
  if (pc.size == 1 && !envFlag("CUDA_FORCE_KERNELS", false)) {
    localCast(pc, static_cast<const char*>(in.local) + inOffset, static_cast<char*>(out.local) + outOffset, count, dt,
              outDt, op, scale, stream, "allreduceCast(local)");
    return;
  }
  const bool vec = in.vectorOk && out.vectorOk && inOffset % 32 == 0 && outOffset % 32 == 0;
  const bool useMc = in.mc != nullptr && vec && pc.size > 2 && nvlsSupports(dt, op) &&
                     count * elementSize(dt) >= tuning().nvlsMinBytes;
  const void* kernel = castKernelFor(dt, outDt);
  const int wanted = ep.blocks > 0 ? ep.blocks : tuning().maxBlocks;
  const int blocks = clampBlocks(pc, kernel, wanted, ceilDiv(count, size_t(8)) / pc.size, 1);
  prologue(pc, stream);
  launchCastAllreduce(pc.comm(), in.ptrsAt(inOffset), useMc ? static_cast<char*>(in.mc) + inOffset : nullptr,
                      out.ptrsAt(outOffset), count, dt, outDt, op, scale, vec, blocks, stream);
  finish(pc, stream, "allreduceCast");
}


// ---- data movement ---------------------------------------------------------------------

namespace {

std::vector<size_t> prefix(const std::vector<size_t>& v) {
  std::vector<size_t> off(v.size() + 1, 0);
  for (size_t i = 0; i < v.size(); i++) off[i + 1] = off[i] + v[i];
  return off;
}

// A view of the pool's bulk region as a PeerBuffer-like target for staged calls.
struct StagedOut {
  PeerPtrs ptrs;
  void* mc;
  char* mine;
};

StagedOut stagedBulk(const PeerContext& pc, size_t needBytes, const char* what) {
  const auto l = layoutOf(pc);
  GLB_ENFORCE_LE(needBytes, l.bulkBytes, what, ": ", needBytes,
                 " bytes do not fit the staging pool; register the buffer (PeerContext::registerBuffer / "
                 "allocSymmetric) or raise GLB_CUDA_STAGE_MB");
  StagedOut s;
  s.ptrs = pc.stagePtrs(l.bulkOff);
  s.mc = pc.stageMc(l.bulkOff);
  s.mine = static_cast<char*>(s.ptrs.p[pc.rank]);
  return s;
}

// Store-only kernels (broadcast / gather / alltoall pushes) are light on registers, so two
// CTAs per SM stay co-resident: their cap is 2x the reduce kernels'.
// Grid of a store-only kernel: enough CTAs for `workBytes`, at most what the tuning table (keyed
// by `keyBytes`) or the copyBlocks knob allows, and never more than can be co-resident for THIS
// kernel (occupancy query: every CTA waits for its twin on the peers, so all must be running).
int bwBlocks(PeerContext& pc, const char* coll, const void* kernel, size_t workBytes, size_t keyBytes = ~size_t(0)) {
  if (keyBytes == ~size_t(0)) keyBytes = workBytes;
  size_t want = ceilDiv(std::max<size_t>(workBytes / 16, 1), static_cast<size_t>(kThreads) * 4);
  const int resident = kernel != nullptr ? pc.coResidentBlocks(kernel) : pc.maxBlocks();
  int cap = std::min({tuning().copyBlocks, resident, kMaxBlocks});
  if (const TuneEntry* e = TuningTable::get().lookup(coll, pc.size, BufKind::REGISTERED, keyBytes)) {
    if (e->blocks > 0) cap = std::min({e->blocks, resident, kMaxBlocks});
  }
  return std::max(1, static_cast<int>(std::min<size_t>(want, static_cast<size_t>(cap))));
}

}  // namespace

namespace {
// Launch shape of one broadcast kernel. mode 0 = root pushes everything, 1 = scatter +
// allgather, 2 = multimem.st, 3 = chunk-pipelined relay (see broadcastKernel).
struct BcastShape {
  int mode = 0;
  int blocks = 1;
  int tile = 0;
};

BcastShape planBroadcast(PeerContext& pc, size_t bytes, bool vec, bool hasMc) {
  const auto& t = tuning();
  BcastShape sh;
  const TuneEntry* e = TuningTable::get().lookup("broadcast", pc.size, BufKind::REGISTERED, bytes);
  // multimem.st pays off when the root would otherwise send P-1 copies: P > 2. From
  // bcastRelayMinBytes up the pipelined relay keeps every link busy instead.
  if (pc.size > 2 && vec && bytes >= t.bcastRelayMinBytes) {
    sh.mode = 3;
  } else if (hasMc && vec && pc.size > 2 && bytes >= t.bcastDirectMaxBytes) {
    sh.mode = 2;
  } else if (bytes > t.bcastDirectMaxBytes && pc.size > 2) {
    sh.mode = 1;
  }
  if (e != nullptr) {
    if (e->algo == "relay" && vec && pc.size > 2) sh.mode = 3;
    if (e->algo == "nvls" && hasMc && vec) sh.mode = 2;
    if (e->algo == "scatter" && pc.size > 2) sh.mode = 1;
    if (e->algo == "direct") sh.mode = 0;
  }
  long forced = envInt("CUDA_BCAST_MODE", -1);
  if (forced >= 0 && forced <= 3 && (forced != 2 || (hasMc && vec)) && (forced != 3 || (vec && pc.size > 2))) {
    sh.mode = static_cast<int>(forced);
  }
  sh.blocks = bwBlocks(pc, "broadcast", broadcastKernelPtr(), sh.mode == 1 ? bytes / pc.size * 2 : bytes, bytes);
  if (sh.mode == 3) {
    // Tiles of at least 8 KB per CTA (one full pass of the CTA), at least ~4 chunks in flight
    // behind each other; small payloads use fewer CTAs rather than smaller tiles.
    const size_t units = bytes / 16;
    const size_t R = static_cast<size_t>(pc.size - 1);
    long tile = envInt("CUDA_BCAST_TILE", e != nullptr && e->tile > 0 ? e->tile : 0);
    if (tile <= 0) {
      tile = 512;
      while (tile < 4096 && units / (R * static_cast<size_t>(sh.blocks) * static_cast<size_t>(tile) * 2) >= 8) tile *= 2;
    }
    sh.tile = static_cast<int>(tile);
    const size_t fit = std::max<size_t>(units / (R * static_cast<size_t>(sh.tile) * 4), 1);
    sh.blocks = static_cast<int>(std::min<size_t>(static_cast<size_t>(sh.blocks), fit));
  }
  return sh;
}
}  // namespace

void broadcast(PeerContext& pc, const PeerBuffer& buf, size_t byteOffset, size_t bytes, int root,
               cudaStream_t stream) {
  GLB_TRACE_RANGE("glb::cuda::broadcast");
  if (bytes == 0 || pc.size == 1) return;
  GLB_ENFORCE(root >= 0 && root < pc.size, "broadcast: invalid root ", root);
  GLB_ENFORCE_LE(byteOffset + bytes, buf.bytes, "broadcast range exceeds the registered buffer");
  DeviceGuard g(pc.device);
  const bool vec = buf.vectorOk && byteOffset % 16 == 0;
  const BcastShape sh = planBroadcast(pc, bytes, vec, buf.mc != nullptr);
  prologue(pc, stream);
  launchBroadcast(pc.comm(), buf.ptrsAt(byteOffset), buf.mc ? static_cast<char*>(buf.mc) + byteOffset : nullptr,
                  bytes, root, sh.mode, vec, sh.blocks, sh.tile, stream);
  finish(pc, stream, "broadcast");
}

void broadcast(PeerContext& pc, void* ptr, size_t bytes, int root, cudaStream_t stream) {
  GLB_TRACE_RANGE("glb::cuda::broadcast(staged)");
  if (bytes == 0 || pc.size == 1) return;
  DeviceGuard g(pc.device);
  const auto l = layoutOf(pc);
  const size_t piece = l.bulkBytes / 16 * 16;
  PeerPtrs stage = pc.stagePtrs(l.bulkOff);
  char* mine = static_cast<char*>(stage.p[pc.rank]);
  for (size_t done = 0; done < bytes; done += piece) {
    const size_t n = std::min(piece, bytes - done);
    char* p = static_cast<char*>(ptr) + done;
    if (pc.rank == root) GLB_CUDA_CHECK(cudaMemcpyAsync(mine, p, n, cudaMemcpyDeviceToDevice, stream));
    const BcastShape sh = planBroadcast(pc, n, true, pc.nvlsAvailable());
    prologue(pc, stream);
    launchBroadcast(pc.comm(), stage, pc.stageMc(l.bulkOff), n, root, sh.mode, true, sh.blocks, sh.tile, stream);
    finish(pc, stream, "broadcast(staged)");
    if (pc.rank != root) GLB_CUDA_CHECK(cudaMemcpyAsync(p, mine, n, cudaMemcpyDeviceToDevice, stream));
  }
}

namespace {
void gatherCommon(PeerContext& pc, const void* in, const PeerPtrs& outs, void* mcOut, bool vecOut,
                  const std::vector<size_t>& bytesPerRank, int onlyDst, cudaStream_t stream) {
  GLB_TRACE_RANGE("glb::cuda::allgather/gather");
  GLB_ENFORCE_EQ(static_cast<int>(bytesPerRank.size()), pc.size, "need one byte count per rank");
  auto off = prefix(bytesPerRank);
  const bool vec = vecOut && reinterpret_cast<uintptr_t>(in) % 16 == 0;
  // The barrier pairs CTA b with CTA b of every peer: the grid must be the same on every
  // rank, so it is sized from the LARGEST block (every rank holds the whole size vector).
  const size_t largest = *std::max_element(bytesPerRank.begin(), bytesPerRank.end());
  prologue(pc, stream);
  launchGatherPush(pc.comm(), in, outs, mcOut, off.data(), bytesPerRank.data(), onlyDst, vec,
                   bwBlocks(pc, "allgather", gatherPushKernelPtr(), largest), stream);
  finish(pc, stream, "allgather/gather");
}

bool allEqual(const std::vector<size_t>& v) {
  for (size_t x : v) {
    if (x != v[0]) return false;
  }
  return true;
}

// Small uniform allgather / alltoall: flag-in-data lines, no barrier, any output pointer.
bool tryLLExchange(PeerContext& pc, const void* in, void* outLocal, size_t bytesPerBlock, int mode,
                   cudaStream_t stream) {
  size_t limit = std::min(tuning().llMaxBytes, pc.llMaxBytes());
  if (const TuneEntry* e = TuningTable::get().lookup(mode == 0 ? "allgather" : "alltoall", pc.size, BufKind::REGISTERED,
                                                     bytesPerBlock)) {
    if (e->algo != "ll") return false;
    limit = pc.llMaxBytes();
  }
  if (bytesPerBlock == 0 || bytesPerBlock > limit || envFlag("CUDA_LL_DISABLE", false)) return false;
  const size_t units = ceilDiv(bytesPerBlock, size_t(8)) * pc.size;
  int threads = static_cast<int>(std::min<size_t>(kThreads, roundUp(std::max<size_t>(units, 32), 32)));
  int blocks = static_cast<int>(std::min<size_t>(ceilDiv(units, static_cast<size_t>(threads)), 16));
  blocks = std::max(1, std::min(blocks, pc.maxBlocks()));
  prologue(pc, stream);
  launchLLExchange(pc.comm(), in, outLocal, bytesPerBlock, mode, pc.llPtrs(), pc.llSrcStride(), pc.llParityStride(), blocks,
                   threads, stream);
  finish(pc, stream, "ll exchange");
  return true;
}
}  // namespace

void allgatherv(PeerContext& pc, const void* in, const PeerBuffer& out, size_t outOffset,
                const std::vector<size_t>& bytesPerRank, cudaStream_t stream) {
  DeviceGuard g(pc.device);
  auto off = prefix(bytesPerRank);
  GLB_ENFORCE_LE(outOffset + off.back(), out.bytes, "allgather output exceeds the registered buffer");
  if (pc.size == 1) {
    char* dst = static_cast<char*>(out.local) + outOffset;
    if (dst != in && off.back() > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(dst, in, off.back(), cudaMemcpyDeviceToDevice, stream));
    return;
  }
  if (allEqual(bytesPerRank) &&
      tryLLExchange(pc, in, static_cast<char*>(out.local) + outOffset, bytesPerRank[0], 0, stream)) {
    return;
  }
  // No multicast here: an allgather's bottleneck is what every GPU RECEIVES ((P-1)/P of the
  // output either way); multimem.st would only relieve the uplink and additionally deliver
  // each block back to its sender (measured at P=2: 312 GB/s with, 540 GB/s without).
  gatherCommon(pc, in, out.ptrsAt(outOffset), nullptr, out.vectorOk && outOffset % 16 == 0, bytesPerRank, -1, stream);
}

void allgatherv(PeerContext& pc, const void* in, void* out, const std::vector<size_t>& bytesPerRank,
                cudaStream_t stream) {
  DeviceGuard g(pc.device);
  auto off = prefix(bytesPerRank);
  if (pc.size == 1) {
    if (out != in && off.back() > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(out, in, off.back(), cudaMemcpyDeviceToDevice, stream));
    return;
  }
  if (allEqual(bytesPerRank) && tryLLExchange(pc, in, out, bytesPerRank[0], 0, stream)) return;
  auto st = stagedBulk(pc, off.back(), "allgather");
  gatherCommon(pc, in, st.ptrs, nullptr, true, bytesPerRank, -1, stream);
  if (off.back() > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(out, st.mine, off.back(), cudaMemcpyDeviceToDevice, stream));
}

namespace {
std::vector<size_t> bytesOf(const std::vector<size_t>& counts, DataType dt) {
  std::vector<size_t> b(counts);
  for (size_t& x : b) x *= elementSize(dt);
  return b;
}

void checkCast(DataType in, DataType out, const char* what) {
  GLB_ENFORCE(castSupported(in, out), what, ": supported conversions are f32 -> f16 / bf16 and f16 / bf16 -> f32");
}

// No LL variant and no multicast: the push kernel with a conversion, grid from the largest
// block's OUTPUT bytes (the "allgather" table entry), identical on every rank.
void gatherCastCommon(PeerContext& pc, const void* in, DataType inDt, const PeerPtrs& outs, bool vecOut,
                      const std::vector<size_t>& counts, DataType outDt, cudaStream_t stream) {
  GLB_TRACE_RANGE("glb::cuda::allgatherCast");
  auto off = prefix(counts);
  const size_t largest = *std::max_element(counts.begin(), counts.end());
  const bool vec = vecOut && reinterpret_cast<uintptr_t>(in) % 16 == 0;
  const int blocks = bwBlocks(pc, "allgather", gatherPushCastKernelFor(inDt, outDt), largest * elementSize(outDt));
  prologue(pc, stream);
  launchGatherPushCast(pc.comm(), in, outs, off.data(), counts.data(), inDt, outDt, vec, blocks, stream);
  finish(pc, stream, "allgatherCast");
}
}  // namespace

void allgathervCast(PeerContext& pc, const void* in, DataType inDt, const PeerBuffer& out, size_t outOffset,
                    const std::vector<size_t>& counts, DataType outDt, cudaStream_t stream) {
  if (inDt == outDt) {
    allgatherv(pc, in, out, outOffset, bytesOf(counts, inDt), stream);
    return;
  }
  checkCast(inDt, outDt, "allgatherCast");
  GLB_ENFORCE_EQ(static_cast<int>(counts.size()), pc.size, "need one element count per rank");
  DeviceGuard g(pc.device);
  auto off = prefix(counts);
  GLB_ENFORCE_LE(outOffset + off.back() * elementSize(outDt), out.bytes, "allgather output exceeds the registered buffer");
  char* dst = static_cast<char*>(out.local) + outOffset;
  if (pc.size == 1) {
    localCast(pc, in, dst, counts[0], inDt, outDt, ReduceOp::SUM, 1.0f, stream, "allgatherCast(local)");
    return;
  }
  gatherCastCommon(pc, in, inDt, out.ptrsAt(outOffset), out.vectorOk && outOffset % 16 == 0, counts, outDt, stream);
}

void allgathervCast(PeerContext& pc, const void* in, DataType inDt, void* out, const std::vector<size_t>& counts,
                    DataType outDt, cudaStream_t stream) {
  if (inDt == outDt) {
    allgatherv(pc, in, out, bytesOf(counts, inDt), stream);
    return;
  }
  checkCast(inDt, outDt, "allgatherCast");
  GLB_ENFORCE_EQ(static_cast<int>(counts.size()), pc.size, "need one element count per rank");
  DeviceGuard g(pc.device);
  if (pc.size == 1) {
    localCast(pc, in, out, counts[0], inDt, outDt, ReduceOp::SUM, 1.0f, stream, "allgatherCast(local)");
    return;
  }
  const size_t outBytes = prefix(counts).back() * elementSize(outDt);
  auto st = stagedBulk(pc, outBytes, "allgather");
  gatherCastCommon(pc, in, inDt, st.ptrs, true, counts, outDt, stream);
  if (outBytes > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(out, st.mine, outBytes, cudaMemcpyDeviceToDevice, stream));
}

void gatherv(PeerContext& pc, const void* in, const PeerBuffer& out, size_t outOffset,
             const std::vector<size_t>& bytesPerRank, int root, cudaStream_t stream) {
  DeviceGuard g(pc.device);
  GLB_ENFORCE(root >= 0 && root < pc.size, "gather: invalid root ", root);
  if (pc.size == 1) {
    char* dst = static_cast<char*>(out.local) + outOffset;
    if (dst != in && bytesPerRank[0] > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(dst, in, bytesPerRank[0], cudaMemcpyDeviceToDevice, stream));
    return;
  }
  gatherCommon(pc, in, out.ptrsAt(outOffset), nullptr, out.vectorOk && outOffset % 16 == 0, bytesPerRank, root, stream);
}

void gatherv(PeerContext& pc, const void* in, void* out, const std::vector<size_t>& bytesPerRank, int root,
             cudaStream_t stream) {
  DeviceGuard g(pc.device);
  auto off = prefix(bytesPerRank);
  if (pc.size == 1) {
    if (out != in && off.back() > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(out, in, off.back(), cudaMemcpyDeviceToDevice, stream));
    return;
  }
  auto st = stagedBulk(pc, off.back(), "gather");
  gatherCommon(pc, in, st.ptrs, nullptr, true, bytesPerRank, root, stream);
  if (pc.rank == root && off.back() > 0) {
    GLB_CUDA_CHECK(cudaMemcpyAsync(out, st.mine, off.back(), cudaMemcpyDeviceToDevice, stream));
  }
}

namespace {
// `uniform` is a property of the ENTRY POINT (alltoall() vs alltoallv()), never derived from
// this rank's own tables: ranks of one alltoallv call may hold tables that look uniform
// locally while a peer's do not, and they must all run the same protocol. The v-variant
// therefore always exchanges receive offsets through the signal pads and always launches
// the same fixed grid (its byte counts are rank-local, the grid must not be).
void alltoallCommon(PeerContext& pc, const void* in, const std::vector<size_t>& sendBytes, const PeerPtrs& outs,
                    bool vecOut, const std::vector<size_t>& recvBytes, bool uniform, cudaStream_t stream) {
  GLB_TRACE_RANGE("glb::cuda::alltoall");
  GLB_ENFORCE_EQ(static_cast<int>(sendBytes.size()), pc.size, "alltoall: need one send size per rank");
  GLB_ENFORCE_EQ(static_cast<int>(recvBytes.size()), pc.size, "alltoall: need one recv size per rank");
  auto soff = prefix(sendBytes);
  auto roff = prefix(recvBytes);
  // dstOff[j] = where my chunk lands in rank j's output = rank j's receive offset
  // for source `me`. For the uniform case that is me * chunk; for the v-variant the
  // kernel reads it from rank j's pad (published there before the first barrier).
  std::vector<size_t> dstOff(pc.size);
  for (int j = 0; j < pc.size; j++) dstOff[j] = uniform ? static_cast<size_t>(pc.rank) * sendBytes[0] : ~size_t(0);
  const bool vec = vecOut && reinterpret_cast<uintptr_t>(in) % 16 == 0;
  int blocks;
  if (uniform) {
    blocks = bwBlocks(pc, "alltoall", alltoallPushKernelPtr(), soff.back(), sendBytes[0]);
  } else {
    blocks = std::max(1, std::min({tuning().alltoallvBlocks, pc.coResidentBlocks(alltoallPushKernelPtr()), kMaxBlocks}));
  }
  prologue(pc, stream);
  launchAlltoallPush(pc.comm(), in, outs, soff.data(), sendBytes.data(), dstOff.data(), uniform ? nullptr : roff.data(),
                     -1, vec, blocks, stream);
  finish(pc, stream, "alltoall");
}
}  // namespace

void alltoall(PeerContext& pc, const void* in, const PeerBuffer& out, size_t outOffset, size_t bytes,
              cudaStream_t stream) {
  DeviceGuard g(pc.device);
  GLB_ENFORCE_LE(outOffset + bytes * pc.size, out.bytes, "alltoall output exceeds the registered buffer");
  char* dst = static_cast<char*>(out.local) + outOffset;
  if (pc.size == 1) {
    if (dst != in && bytes > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(dst, in, bytes, cudaMemcpyDeviceToDevice, stream));
    return;
  }
  if (tryLLExchange(pc, in, dst, bytes, 1, stream)) return;
  std::vector<size_t> sizes(pc.size, bytes);
  alltoallCommon(pc, in, sizes, out.ptrsAt(outOffset), out.vectorOk && outOffset % 16 == 0, sizes, true, stream);
}

void alltoall(PeerContext& pc, const void* in, void* out, size_t bytes, cudaStream_t stream) {
  DeviceGuard g(pc.device);
  if (pc.size == 1) {
    if (out != in && bytes > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(out, in, bytes, cudaMemcpyDeviceToDevice, stream));
    return;
  }
  if (tryLLExchange(pc, in, out, bytes, 1, stream)) return;
  auto st = stagedBulk(pc, bytes * pc.size, "alltoall");
  std::vector<size_t> sizes(pc.size, bytes);
  alltoallCommon(pc, in, sizes, st.ptrs, true, sizes, true, stream);
  if (bytes > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(out, st.mine, bytes * pc.size, cudaMemcpyDeviceToDevice, stream));
}

void alltoallv(PeerContext& pc, const void* in, const std::vector<size_t>& sendBytes, const PeerBuffer& out,
               size_t outOffset, const std::vector<size_t>& recvBytes, cudaStream_t stream) {
  DeviceGuard g(pc.device);
  auto roff = prefix(recvBytes);
  GLB_ENFORCE_LE(outOffset + roff.back(), out.bytes, "alltoall output exceeds the registered buffer");
  if (pc.size == 1) {
    char* dst = static_cast<char*>(out.local) + outOffset;
    if (dst != in && sendBytes[0] > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(dst, in, sendBytes[0], cudaMemcpyDeviceToDevice, stream));
    return;
  }
  alltoallCommon(pc, in, sendBytes, out.ptrsAt(outOffset), out.vectorOk && outOffset % 16 == 0, recvBytes, false, stream);
}

void alltoallv(PeerContext& pc, const void* in, const std::vector<size_t>& sendBytes, void* out,
               const std::vector<size_t>& recvBytes, cudaStream_t stream) {
  DeviceGuard g(pc.device);
  auto roff = prefix(recvBytes);
  if (pc.size == 1) {
    if (out != in && sendBytes[0] > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(out, in, sendBytes[0], cudaMemcpyDeviceToDevice, stream));
    return;
  }
  // Every rank stages the same span so the (data-dependent) fit check cannot diverge.
  auto st = stagedBulk(pc, roff.back(), "alltoall");
  alltoallCommon(pc, in, sendBytes, st.ptrs, true, recvBytes, false, stream);
  if (roff.back() > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(out, st.mine, roff.back(), cudaMemcpyDeviceToDevice, stream));
}

void scatter(PeerContext& pc, const void* in, const PeerBuffer& out, size_t outOffset, size_t bytes, int root,
             cudaStream_t stream) {
  DeviceGuard g(pc.device);
  GLB_ENFORCE(root >= 0 && root < pc.size, "scatter: invalid root ", root);
  GLB_ENFORCE_LE(outOffset + bytes, out.bytes, "scatter output exceeds the registered buffer");
  if (pc.size == 1) {
    char* dst = static_cast<char*>(out.local) + outOffset;
    if (dst != in && bytes > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(dst, in, bytes, cudaMemcpyDeviceToDevice, stream));
    return;
  }
  std::vector<size_t> soff(pc.size), slen(pc.size, bytes), doff(pc.size, 0);
  for (int j = 0; j < pc.size; j++) soff[j] = static_cast<size_t>(j) * bytes;
  const bool vec = out.vectorOk && outOffset % 16 == 0 && (pc.rank != root || reinterpret_cast<uintptr_t>(in) % 16 == 0);
  prologue(pc, stream);
  launchAlltoallPush(pc.comm(), in, out.ptrsAt(outOffset), soff.data(), slen.data(), doff.data(), nullptr, root, vec,
                     bwBlocks(pc, "alltoall", alltoallPushKernelPtr(), bytes * pc.size, bytes), stream);
  finish(pc, stream, "scatter");
}

void scatter(PeerContext& pc, const void* in, void* out, size_t bytes, int root, cudaStream_t stream) {
  DeviceGuard g(pc.device);
  if (pc.size == 1) {
    if (out != in && bytes > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(out, in, bytes, cudaMemcpyDeviceToDevice, stream));
    return;
  }
  auto st = stagedBulk(pc, bytes, "scatter");
  std::vector<size_t> soff(pc.size), slen(pc.size, bytes), doff(pc.size, 0);
  for (int j = 0; j < pc.size; j++) soff[j] = static_cast<size_t>(j) * bytes;
  prologue(pc, stream);
  launchAlltoallPush(pc.comm(), in, st.ptrs, soff.data(), slen.data(), doff.data(), nullptr, root,
                     pc.rank != root || reinterpret_cast<uintptr_t>(in) % 16 == 0,
                     bwBlocks(pc, "alltoall", alltoallPushKernelPtr(), bytes * pc.size, bytes), stream);
  finish(pc, stream, "scatter(staged)");
  if (bytes > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(out, st.mine, bytes, cudaMemcpyDeviceToDevice, stream));
}

namespace {
void reducePullCommon(PeerContext& pc, const PeerPtrs& ins, void* mcIn, bool vecIn, void* out,
                      const std::vector<size_t>& counts, DataType dt, ReduceOp op, double scaleD, cudaStream_t stream) {
  GLB_TRACE_RANGE("glb::cuda::reduce_scatter/reduce");
  GLB_ENFORCE_EQ(static_cast<int>(counts.size()), pc.size, "need one element count per rank");
  GLB_ENFORCE(op != ReduceOp::CUSTOM, "custom reductions run on the host path only");
  auto off = prefix(counts);
  const size_t es = elementSize(dt);
  // In-switch reduction only for P > 2 (at P = 2 it doubles the uplink traffic).
  // Decisions that shape the launch use the LARGEST share: identical on every rank.
  const size_t largest = *std::max_element(counts.begin(), counts.end());
  bool wantMc = tuning().nvlsReduceScatter;
  int cap = tuning().maxBlocks;
  if (const TuneEntry* e = TuningTable::get().lookup("reduce_scatter", pc.size, mcIn ? BufKind::SYMMETRIC : BufKind::REGISTERED,
                                                     largest * es)) {
    wantMc = e->algo == "nvls";
    if (e->blocks > 0) cap = e->blocks;
  }
  const bool useMc = mcIn != nullptr && pc.size > 2 && wantMc && nvlsSupports(dt, op) && largest * es >= tuning().nvlsMinBytes;
  Epilogue ep;
  ep.scale = scaleD;
  const float scale = scaleOf(ep, dt);
  prologue(pc, stream);
  launchReducePull(pc.comm(), ins, mcIn, out, off.data(), counts.data(), dt, op, scale, vecIn, useMc,
                   std::min(blocksFor(pc, largest * es / 16, 1, cap), pc.coResidentBlocks(reducePullKernelPtr(dt, pc.size))),
                   stream);
  finish(pc, stream, "reduce_scatter");
}
}  // namespace

namespace {
// Small reduce_scatter with equal shares: flag-in-data lines, no barrier, any input pointer.
bool tryLLReduceScatter(PeerContext& pc, const void* in, void* out, const std::vector<size_t>& counts, DataType dt,
                        ReduceOp op, double scaleD, cudaStream_t stream) {
  if (pc.size < 2 || !allEqual(counts) || counts[0] == 0 || envFlag("CUDA_LL_DISABLE", false)) return false;
  const size_t bytes = counts[0] * elementSize(dt);
  size_t limit = std::min(tuning().llMaxBytes, pc.llMaxBytes());
  if (const TuneEntry* e = TuningTable::get().lookup("reduce_scatter", pc.size, BufKind::REGISTERED, bytes)) {
    if (e->algo != "ll") return false;
    limit = pc.llMaxBytes();
  }
  if (bytes > limit) return false;
  Epilogue ep;
  ep.scale = scaleD;
  const float scale = scaleOf(ep, dt);
  const size_t units = ceilDiv(bytes, size_t(8)) * pc.size;
  int threads = static_cast<int>(std::min<size_t>(kThreads, roundUp(std::max<size_t>(units, 32), 32)));
  int blocks = static_cast<int>(std::min<size_t>(ceilDiv(units, static_cast<size_t>(threads)), 16));
  prologue(pc, stream);
  launchLLReduceScatter(pc.comm(), in, out, counts[0], dt, op, scale, pc.llPtrs(), pc.llSrcStride(), pc.llParityStride(),
                        std::max(1, blocks), threads, stream);
  finish(pc, stream, "reduce_scatter(ll)");
  return true;
}
}  // namespace

void reduce_scatter(PeerContext& pc, const PeerBuffer& in, size_t inOffset, void* out,
                    const std::vector<size_t>& counts, DataType dt, ReduceOp op, cudaStream_t stream, double scale) {
  DeviceGuard g(pc.device);
  auto off = prefix(counts);
  const size_t es = elementSize(dt);
  GLB_ENFORCE_LE(inOffset + off.back() * es, in.bytes, "reduce_scatter input exceeds the registered buffer");
  if (pc.size == 1) {
    const char* src = static_cast<const char*>(in.local) + inOffset;
    if (src != out && counts[0] > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(out, src, counts[0] * es, cudaMemcpyDeviceToDevice, stream));
    return;
  }
  GLB_ENFORCE(op != ReduceOp::CUSTOM, "custom reductions run on the host path only");
  if (tryLLReduceScatter(pc, static_cast<const char*>(in.local) + inOffset, out, counts, dt, op, scale, stream)) return;
  reducePullCommon(pc, in.ptrsAt(inOffset), in.mc ? static_cast<char*>(in.mc) + inOffset : nullptr,
                   in.vectorOk && inOffset % 16 == 0, out, counts, dt, op, scale, stream);
}

void reduce_scatter(PeerContext& pc, const void* in, void* out, const std::vector<size_t>& counts, DataType dt,
                    ReduceOp op, cudaStream_t stream, double scale) {
  DeviceGuard g(pc.device);
  auto off = prefix(counts);
  const size_t es = elementSize(dt);
  if (pc.size == 1) {
    if (in != out && counts[0] > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(out, in, counts[0] * es, cudaMemcpyDeviceToDevice, stream));
    return;
  }
  GLB_ENFORCE(op != ReduceOp::CUSTOM, "custom reductions run on the host path only");
  if (tryLLReduceScatter(pc, in, out, counts, dt, op, scale, stream)) return;
  auto st = stagedBulk(pc, off.back() * es, "reduce_scatter");
  if (off.back() > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(st.mine, in, off.back() * es, cudaMemcpyDeviceToDevice, stream));
  reducePullCommon(pc, st.ptrs, st.mc, true, out, counts, dt, op, scale, stream);
}

namespace {
// The pull kernel with a conversion. Grid from the "reduce_scatter" table entry keyed by the
// largest share's INPUT bytes, as reducePullCommon sizes it; the kernel reads peers directly,
// so the entry for registered buffers applies whether or not the input has a multicast alias.
void reducePullCastCommon(PeerContext& pc, const PeerPtrs& ins, bool vecIn, void* out, const std::vector<size_t>& counts,
                          DataType dt, DataType outDt, ReduceOp op, float scale, cudaStream_t stream) {
  GLB_TRACE_RANGE("glb::cuda::reduceScatterCast");
  auto off = prefix(counts);
  const size_t inBytes = *std::max_element(counts.begin(), counts.end()) * elementSize(dt);
  int cap = tuning().maxBlocks;
  if (const TuneEntry* e = TuningTable::get().lookup("reduce_scatter", pc.size, BufKind::REGISTERED, inBytes)) {
    if (e->blocks > 0) cap = e->blocks;
  }
  const int blocks =
      std::min(blocksFor(pc, inBytes / 16, 1, cap), pc.coResidentBlocks(reducePullCastKernelFor(dt, outDt, pc.size)));
  prologue(pc, stream);
  launchReducePullCast(pc.comm(), ins, out, off.data(), counts.data(), dt, outDt, op, scale, vecIn, blocks, stream);
  finish(pc, stream, "reduceScatterCast");
}

// Checks shared by both reduceScatterCast overloads; returns the scale as the kernels take it.
float reduceScatterCastArgs(PeerContext& pc, const std::vector<size_t>& counts, DataType dt, DataType outDt,
                            ReduceOp op, double scaleD) {
  checkCast(dt, outDt, "reduceScatterCast");
  GLB_ENFORCE(op != ReduceOp::CUSTOM, "custom reductions run on the host path only");
  GLB_ENFORCE_EQ(static_cast<int>(counts.size()), pc.size, "need one element count per rank");
  Epilogue ep;
  ep.scale = scaleD;
  return scaleOf(ep, DataType::FLOAT32);
}
}  // namespace

void reduceScatterCast(PeerContext& pc, const PeerBuffer& in, size_t inOffset, void* out,
                       const std::vector<size_t>& counts, DataType dt, DataType outDt, ReduceOp op,
                       cudaStream_t stream, double scaleD) {
  if (dt == outDt) {
    reduce_scatter(pc, in, inOffset, out, counts, dt, op, stream, scaleD);
    return;
  }
  const float scale = reduceScatterCastArgs(pc, counts, dt, outDt, op, scaleD);
  DeviceGuard g(pc.device);
  auto off = prefix(counts);
  GLB_ENFORCE_LE(inOffset + off.back() * elementSize(dt), in.bytes, "reduce_scatter input exceeds the registered buffer");
  const char* src = static_cast<const char*>(in.local) + inOffset;
  // A single rank converts locally in every overload, like reduce_scatter / allgatherv, which
  // copy locally whatever GLB_CUDA_FORCE_KERNELS says.
  if (pc.size == 1) {
    localCast(pc, src, out, counts[0], dt, outDt, op, scale, stream, "reduceScatterCast(local)");
    return;
  }
  reducePullCastCommon(pc, in.ptrsAt(inOffset), in.vectorOk && inOffset % 16 == 0, out, counts, dt, outDt, op, scale,
                       stream);
}

void reduceScatterCast(PeerContext& pc, const void* in, void* out, const std::vector<size_t>& counts, DataType dt,
                       DataType outDt, ReduceOp op, cudaStream_t stream, double scaleD) {
  if (dt == outDt) {
    reduce_scatter(pc, in, out, counts, dt, op, stream, scaleD);
    return;
  }
  const float scale = reduceScatterCastArgs(pc, counts, dt, outDt, op, scaleD);
  DeviceGuard g(pc.device);
  if (pc.size == 1) {
    localCast(pc, in, out, counts[0], dt, outDt, op, scale, stream, "reduceScatterCast(local)");
    return;
  }
  const size_t inBytes = prefix(counts).back() * elementSize(dt);
  auto st = stagedBulk(pc, inBytes, "reduce_scatter");
  if (inBytes > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(st.mine, in, inBytes, cudaMemcpyDeviceToDevice, stream));
  reducePullCastCommon(pc, st.ptrs, true, out, counts, dt, outDt, op, scale, stream);
}

void reduce(PeerContext& pc, const PeerBuffer& in, size_t inOffset, const PeerBuffer& out, size_t outOffset,
            size_t count, DataType dt, ReduceOp op, int root, cudaStream_t stream) {
  DeviceGuard g(pc.device);
  GLB_ENFORCE(root >= 0 && root < pc.size, "reduce: invalid root ", root);
  const size_t es = elementSize(dt);
  GLB_ENFORCE_LE(inOffset + count * es, in.bytes, "reduce input exceeds the registered buffer");
  if (pc.size == 1) {
    const char* src = static_cast<const char*>(in.local) + inOffset;
    char* dst = static_cast<char*>(out.local) + outOffset;
    if (src != dst && count > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(dst, src, count * es, cudaMemcpyDeviceToDevice, stream));
    return;
  }
  GLB_ENFORCE(out.peer[root] != nullptr, "reduce: the root's output is not registered");
  // Each rank reduces an equal slice and stores it straight into the root's output.
  std::vector<size_t> counts(pc.size);
  for (int r = 0; r < pc.size; r++) counts[r] = count / pc.size + (static_cast<size_t>(r) < count % pc.size ? 1 : 0);
  auto off = prefix(counts);
  char* dst = static_cast<char*>(out.peer[root]) + outOffset + off[pc.rank] * es;
  reducePullCommon(pc, in.ptrsAt(inOffset), in.mc ? static_cast<char*>(in.mc) + inOffset : nullptr,
                   in.vectorOk && inOffset % 16 == 0, dst, counts, dt, op, 1.0, stream);
}

void reduce(PeerContext& pc, const void* in, void* out, size_t count, DataType dt, ReduceOp op, int root,
            cudaStream_t stream) {
  DeviceGuard g(pc.device);
  const size_t es = elementSize(dt);
  if (pc.size == 1) {
    if (in != out && count > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(out, in, count * es, cudaMemcpyDeviceToDevice, stream));
    return;
  }
  // Stage inputs in the first half of the bulk region, collect results in the second.
  const auto l = layoutOf(pc);
  const size_t half = l.bulkBytes / 2 / 16 * 16;
  GLB_ENFORCE_LE(count * es, half, "reduce: payload does not fit the staging pool; register the buffers");
  PeerPtrs ins = pc.stagePtrs(l.bulkOff);
  PeerPtrs outs = pc.stagePtrs(l.bulkOff + half);
  char* mine = static_cast<char*>(ins.p[pc.rank]);
  if (count > 0) GLB_CUDA_CHECK(cudaMemcpyAsync(mine, in, count * es, cudaMemcpyDeviceToDevice, stream));
  std::vector<size_t> counts(pc.size);
  for (int r = 0; r < pc.size; r++) counts[r] = count / pc.size + (static_cast<size_t>(r) < count % pc.size ? 1 : 0);
  auto off = prefix(counts);
  char* dst = static_cast<char*>(outs.p[root]) + off[pc.rank] * es;
  reducePullCommon(pc, ins, pc.stageMc(l.bulkOff), true, dst, counts, dt, op, 1.0, stream);
  if (pc.rank == root && count > 0) {
    GLB_CUDA_CHECK(cudaMemcpyAsync(out, static_cast<char*>(outs.p[root]), count * es, cudaMemcpyDeviceToDevice, stream));
  }
}

// ---- point to point ------------------------------------------------------------------------------

namespace {
void p2pCommon(PeerContext& pc, const void* sendPtr, size_t sendBytes, int dst, void* recvPtr, size_t recvBytes,
               int src, cudaStream_t stream) {
  GLB_TRACE_RANGE("glb::cuda::p2p");
  DeviceGuard g(pc.device);
  GLB_ENFORCE(sendBytes == 0 || (dst >= 0 && dst < pc.size && dst != pc.rank), "send: invalid destination rank ", dst);
  GLB_ENFORCE(recvBytes == 0 || (src >= 0 && src < pc.size && src != pc.rank), "recv: invalid source rank ", src);
  if (sendBytes == 0 && recvBytes == 0) return;
  pc.checkHealth();
  // No orderStreams / launchGuard: p2p kernels do not use the barrier epoch, and a host
  // rendezvous of ALL ranks would deadlock a pairwise operation.
  const auto& o = pc.options();
  // Both ends must cut a slot into the same stripes: the lane count comes from job-wide
  // values only. Sender and receiver CTAs wait for each other, so they must be co-resident.
  const int lanes = std::max(1, std::min(o.p2pLanes, pc.maxBlocks() / 2));
  launchP2p(pc.comm(), sendPtr, sendBytes, sendBytes ? dst : 0, recvPtr, recvBytes, recvBytes ? src : 0, pc.mailboxPtrs(),
            pc.mailboxStride(), o.p2pSlotBytes, o.p2pSlots, lanes, stream);
  checkLaunch("p2p");
}
}  // namespace

void send(PeerContext& pc, const void* ptr, size_t bytes, int dst, cudaStream_t stream) {
  p2pCommon(pc, ptr, bytes, dst, nullptr, 0, 0, stream);
}

void recv(PeerContext& pc, void* ptr, size_t bytes, int src, cudaStream_t stream) {
  p2pCommon(pc, nullptr, 0, 0, ptr, bytes, src, stream);
}

void sendrecv(PeerContext& pc, const void* sendPtr, size_t sendBytes, int dst, void* recvPtr, size_t recvBytes,
              int src, cudaStream_t stream) {
  p2pCommon(pc, sendPtr, sendBytes, dst, recvPtr, recvBytes, src, stream);
}

void exchange(PeerContext& pc, const void* sendPtr, size_t sendBytes, int dst, const PeerBuffer& recvBuf,
              size_t recvOffset, size_t recvBytes, int src, cudaStream_t stream) {
  GLB_TRACE_RANGE("glb::cuda::exchange");
  DeviceGuard g(pc.device);
  GLB_ENFORCE(sendBytes == 0 || (dst >= 0 && dst < pc.size && dst != pc.rank), "exchange: invalid destination rank ", dst);
  GLB_ENFORCE(recvBytes == 0 || (src >= 0 && src < pc.size && src != pc.rank), "exchange: invalid source rank ", src);
  if (sendBytes == 0 && recvBytes == 0) return;
  GLB_ENFORCE(sendBytes == 0 || recvBuf.peer[dst] != nullptr, "exchange: rank ", dst, " has no mapping of the receive buffer");
  GLB_ENFORCE_LE(recvOffset + std::max(sendBytes, recvBytes), recvBuf.bytes, "exchange: range exceeds the receive buffer");
  pc.checkHealth();
  // Pairwise like send / recv: no barrier epoch, no host rendezvous. The arrival counter
  // counts CTAs, so the grid is a job-wide value.
  const int blocks = std::max(1, std::min(pc.options().exchangeBlocks, pc.maxBlocks()));
  char* remote = sendBytes ? static_cast<char*>(recvBuf.peer[dst]) + recvOffset : nullptr;
  launchExchange(pc.comm(), sendPtr, sendBytes, sendBytes ? dst : 0, remote, recvBytes, recvBytes ? src : 0, blocks,
                 tuning().tmaCopies && std::max(sendBytes, recvBytes) >= 64 * 1024, stream);
  checkLaunch("exchange");
}

void put(PeerContext& pc, const void* local, const PeerBuffer& remote, size_t remoteOffset, size_t bytes, int peer,
         cudaStream_t stream) {
  GLB_ENFORCE(peer >= 0 && peer < pc.size && remote.peer[peer] != nullptr, "put: rank ", peer, " has no mapping of this buffer");
  GLB_ENFORCE_LE(remoteOffset + bytes, remote.bytes, "put: range exceeds the remote buffer");
  if (bytes == 0) return;
  DeviceGuard g(pc.device);
  pc.checkHealth();
  launchPeerCopy(static_cast<char*>(remote.peer[peer]) + remoteOffset, local, bytes, bwBlocks(pc, "put", nullptr, bytes), stream,
                 tuning().tmaCopies);
  checkLaunch("put");
}

void get(PeerContext& pc, void* local, const PeerBuffer& remote, size_t remoteOffset, size_t bytes, int peer,
         cudaStream_t stream) {
  GLB_ENFORCE(peer >= 0 && peer < pc.size && remote.peer[peer] != nullptr, "get: rank ", peer, " has no mapping of this buffer");
  GLB_ENFORCE_LE(remoteOffset + bytes, remote.bytes, "get: range exceeds the remote buffer");
  if (bytes == 0) return;
  DeviceGuard g(pc.device);
  pc.checkHealth();
  launchPeerCopy(local, static_cast<const char*>(remote.peer[peer]) + remoteOffset, bytes, bwBlocks(pc, "get", nullptr, bytes), stream,
                 tuning().tmaCopies);
  checkLaunch("get");
}

}  // namespace cuda
}  // namespace glb
