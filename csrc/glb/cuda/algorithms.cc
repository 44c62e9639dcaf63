#include "glb/cuda/algorithms.h"

#include <map>
#include <mutex>

#include "glb/allreduce.h"
#include "glb/broadcast.h"
#include "glb/common/utils.h"
#include "glb/cuda/kernels.h"
#include "glb/cuda/schedules.h"
#include "glb/cuda/trace.h"

namespace glb {
namespace cuda {

namespace {

// Map the reference's algorithm names to what actually runs. By default the named
// classes resolve per message size (AUTO); literal schedules are opt-in.
AllreduceAlgo effectiveAlgo(AllreduceAlgo requested) {
  switch (requested) {
    case AllreduceAlgo::RING:
    case AllreduceAlgo::RING_CHUNKED:
    case AllreduceAlgo::HALVING_DOUBLING:
    case AllreduceAlgo::BCUBE:
    case AllreduceAlgo::HALVING_DOUBLING_PIPELINED:
      return requested;
    default:
      return requested;
  }
}

std::vector<CudaStream> makeStreams(const std::vector<void*>& ptrs, const std::vector<cudaStream_t>& user) {
  std::vector<CudaStream> out;
  if (!user.empty()) GLB_ENFORCE_EQ(user.size(), ptrs.size(), "need one stream per pointer");
  for (size_t i = 0; i < ptrs.size(); i++) {
    int dev = deviceForPointer(ptrs[i]);
    GLB_ENFORCE_GE(dev, 0, "pointer ", i, " is not a CUDA device pointer");
    if (user.empty()) {
      out.emplace_back(dev);
    } else {
      out.emplace_back(dev, user[i]);
    }
  }
  return out;
}

// All ranks decide together whether the peer path is usable.
}  // namespace

AllreduceAlgo namedAlgo(AllreduceAlgo named) {
  return envFlag("CUDA_LITERAL_SCHEDULES", false) ? named : AllreduceAlgo::AUTO;
}

std::vector<CudaStream> makeStreamsFor(const std::vector<void*>& ptrs, const std::vector<cudaStream_t>& user) {
  return makeStreams(ptrs, user);
}

namespace {
bool peerPathUsable(const std::shared_ptr<Context>& ctx, Workspace ws) {
  if (ws == Workspace::HOST) return false;
  return deviceCount() > 0 && !envFlag("CUDA_FORCE_HOST_WORKSPACE", false);
}
}  // namespace

std::shared_ptr<PeerContext> peerContextFor(const std::shared_ptr<Context>& ctx, int device,
                                            const PeerOptions& optsIfCreated) {
  // The PeerContext is an attachment of the context: it is shared by every algorithm
  // built on that context and dies with it (or at closeConnections()).
  const std::string key = strcat_all("cuda.peer.", device);
  if (auto existing = ctx->getAttachment(key)) return std::static_pointer_cast<PeerContext>(existing);
  // Construction is collective and may block on peers.
  auto pc = std::make_shared<PeerContext>(ctx, device, optsIfCreated);
  ctx->setAttachment(key, pc);
  return pc;
}

void releasePeerContexts(const std::shared_ptr<Context>& ctx) { ctx->clearAttachments(); }

// ---- allreduce ---------------------------------------------------------------------------

struct CudaAllreduceCore::Literal {
  Schedule schedule;
  SchedStep* deviceTable = nullptr;
  int device = 0;
  ~Literal() {
    if (deviceTable != nullptr) {
      DeviceGuard g(device);
      cudaFree(deviceTable);
    }
  }
};

namespace {
bool isLiteral(AllreduceAlgo a) {
  return a == AllreduceAlgo::RING || a == AllreduceAlgo::RING_CHUNKED || a == AllreduceAlgo::HALVING_DOUBLING ||
         a == AllreduceAlgo::BCUBE || a == AllreduceAlgo::HALVING_DOUBLING_PIPELINED;
}
}  // namespace

CudaAllreduceCore::CudaAllreduceCore(std::shared_ptr<Context> ctx, std::vector<void*> ptrs, size_t count,
                                     DataType dt, ReduceOp op, std::vector<cudaStream_t> streams,
                                     AllreduceAlgo algo, Workspace ws)
    : ctx_(std::move(ctx)),
      ptrs_(std::move(ptrs)),
      count_(count),
      dt_(dt),
      op_(op),
      algo_(effectiveAlgo(algo)),
      syncOutputs_(streams.empty()) {
  GLB_ENFORCE(!ptrs_.empty(), "need at least one pointer");
  streams_ = makeStreams(ptrs_, streams);
  const int dev0 = streams_[0].getDeviceID();
  if (ctx_->size > 1 && peerPathUsable(ctx_, ws)) {
    auto pc = peerContextFor(ctx_, dev0);
    if (pc->peerAccessEverywhere()) {
      pc_ = pc;
      reg_ = pc_->resolveBuffer(ptrs_[0], count_ * elementSize(dt_), &regOffset_);
      if (isLiteral(algo_) && count_ > 0) {
        const size_t es = elementSize(dt_);
        const size_t pack = 16 / es;
        auto lit = std::make_unique<Literal>();
        lit->device = dev0;
        AllreduceAlgo a = algo_;
        // The whole-vector ring stages every rank's input in its pool; if that does
        // not fit, the chunked ring is the closest literal schedule.
        if (a == AllreduceAlgo::RING && count_ * es > pc_->stageBytes() / 2) a = AllreduceAlgo::RING_CHUNKED;
        switch (a) {
          case AllreduceAlgo::RING: lit->schedule = buildRingSchedule(ctx_->rank, ctx_->size, count_, pack); break;
          case AllreduceAlgo::RING_CHUNKED:
            lit->schedule = buildRingChunkedSchedule(ctx_->rank, ctx_->size, count_, pack);
            break;
          case AllreduceAlgo::HALVING_DOUBLING:
            lit->schedule = buildHalvingDoublingSchedule(ctx_->rank, ctx_->size, count_, pack);
            break;
          case AllreduceAlgo::HALVING_DOUBLING_PIPELINED:
            lit->schedule = buildHalvingDoublingPipelinedSchedule(ctx_->rank, ctx_->size, count_, pack,
                                                                  static_cast<int>(envInt("CUDA_HD_CHUNKS", 2)));
            break;
          default: lit->schedule = buildBcubeSchedule(ctx_->rank, ctx_->size, count_, ctx_->base, pack); break;
        }
        DeviceGuard g(dev0);
        const size_t tb = lit->schedule.steps.size() * sizeof(SchedStep);
        GLB_CUDA_CHECK(cudaMalloc(reinterpret_cast<void**>(&lit->deviceTable), std::max<size_t>(tb, 16)));
        GLB_CUDA_CHECK(cudaMemcpy(lit->deviceTable, lit->schedule.steps.data(), tb, cudaMemcpyHostToDevice));
        literal_ = std::move(lit);
      }
    }
  }
  // Fold the extra local pointers inside the collective kernel when they live on the same
  // device as the first one (and, across ranks, every pointer is 16-byte aligned so that
  // all ranks pick the same element -> CTA mapping). A single rank needs no alignment: its
  // fused kernel takes unaligned pointers element by element and still rounds once.
  if (ptrs_.size() > 1 && ptrs_.size() - 1 <= static_cast<size_t>(kMaxLocal) && !envFlag("CUDA_NO_LOCAL_FUSION", false)) {
    bool sameDevice = true, aligned = true;
    for (size_t i = 0; i < ptrs_.size(); i++) {
      sameDevice = sameDevice && streams_[i].getDeviceID() == dev0;
      aligned = aligned && reinterpret_cast<uintptr_t>(ptrs_[i]) % 16 == 0;
    }
    if (ctx_->size == 1) {
      fuseLocal_ = sameDevice;
    } else if (pc_ && !literal_) {
      fuseLocal_ = pc_->agree(sameDevice && aligned);
    }
  }
  if (ctx_->size > 1 && !pc_) {
    const size_t bytes = std::max<size_t>(count_ * elementSize(dt_), 16);
    GLB_CUDA_CHECK(cudaMallocHost(&hostScratch_, bytes));
    // Host workspace: cut into chunks so that D2H of chunk c+1, the host collective of chunk c
    // and H2D of chunk c-1 overlap (cuda_allreduce_ring_chunked.cc:129-273 does the same per
    // ring chunk).
    const size_t minChunk = static_cast<size_t>(envInt("CUDA_HOST_CHUNK_MIN", 1 << 20));
    hostChunks_ = static_cast<int>(std::max<size_t>(1, std::min<size_t>(static_cast<size_t>(envInt("CUDA_HOST_CHUNKS", 8)), bytes / minChunk)));
    DeviceGuard g(dev0);
    h2dStream_ = std::make_unique<CudaStream>(dev0);
    chunkEvents_.resize(hostChunks_);
    for (auto& ev : chunkEvents_) GLB_CUDA_CHECK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  }
}

CudaAllreduceCore::~CudaAllreduceCore() {
  if (hostScratch_ != nullptr) cudaFreeHost(hostScratch_);
  for (auto ev : chunkEvents_) cudaEventDestroy(ev);
}

int CudaAllreduceCore::launchesPerRun() const {
  const int cross = ctx_->size > 1 ? 1 : 0;
  if (ptrs_.size() <= 1) return cross;
  if (fuseLocal_) return 1;
  return 2 + cross;
}

// D2H in chunks (all enqueued up front), then per chunk: wait for its copy, run the host
// collective over the transport, enqueue its H2D on a second stream. PCIe down-traffic of
// chunk c+1 and up-traffic of chunk c-1 overlap the network time of chunk c.
void CudaAllreduceCore::runHostWorkspace(CudaStream& s0) {
  const size_t es = elementSize(dt_);
  const size_t per = roundUp(ceilDiv(count_, static_cast<size_t>(hostChunks_)), std::max<size_t>(1, 64 / es));
  char* host = static_cast<char*>(hostScratch_);
  char* dev = static_cast<char*>(ptrs_[0]);
  int n = 0;
  for (size_t lo = 0; lo < count_; lo += per, n++) {
    const size_t len = std::min(per, count_ - lo);
    GLB_CUDA_CHECK(cudaMemcpyAsync(host + lo * es, dev + lo * es, len * es, cudaMemcpyDeviceToHost, *s0));
    GLB_CUDA_CHECK(cudaEventRecord(chunkEvents_[n], *s0));
  }
  ReduceFn fn = getReduceFn(dt_, op_);
  int c = 0;
  for (size_t lo = 0; lo < count_; lo += per, c++) {
    const size_t len = std::min(per, count_ - lo);
    GLB_CUDA_CHECK(cudaEventSynchronize(chunkEvents_[c]));
    AllreduceOptions opts(ctx_);
    opts.setOutputsRaw({host + lo * es}, len, es);
    opts.setReduceFunction([fn](void* o, const void* a, const void* b, size_t k) { fn(o, a, b, k); });
    opts.setTag(0x00CDA000u + static_cast<uint32_t>(c));
    glb::allreduce(opts);
    GLB_CUDA_CHECK(cudaMemcpyAsync(dev + lo * es, host + lo * es, len * es, cudaMemcpyHostToDevice, **h2dStream_));
  }
  h2dStream_->record();
  s0.waitOn(*h2dStream_);
  if (scale_ != 1.0) {
    void* one[1] = {ptrs_[0]};
    launchLocalAllreduceMany(one, 1, count_, dt_, op_, static_cast<float>(scale_), *s0);
    noteLaunch();
  }
}

AllreduceAlgo CudaAllreduceCore::resolvedAlgo() const {
  if (!pc_) return AllreduceAlgo::AUTO;
  if (literal_) return algo_;
  if (algo_ != AllreduceAlgo::AUTO) return algo_;
  return chooseAllreduce(*pc_, count_ * elementSize(dt_), dt_, op_, true, reg_ && reg_->mc != nullptr && regOffset_ % 16 == 0);
}

void CudaAllreduceCore::run() {
  if (count_ == 0) return;
  GLB_TRACE_RANGE("glb::CudaAllreduce::run");
  CudaStream& s0 = streams_[0];
  const size_t bytes = count_ * elementSize(dt_);
  DeviceGuard g(s0.getDeviceID());
  const bool multi = ptrs_.size() > 1;

  if (multi) {
    for (size_t i = 1; i < streams_.size(); i++) {
      streams_[i].record();
      s0.waitOn(streams_[i]);
    }
  }

  Epilogue ep;
  ep.scale = scale_;
  ep.blocks = shapeBlocks_;
  ep.unroll = shapeUnroll_;
  ep.tile = shapeTile_;
  if (fuseLocal_) {
    ep.extra.n = static_cast<int>(ptrs_.size()) - 1;
    for (int k = 0; k < ep.extra.n; k++) ep.extra.p[k] = ptrs_[k + 1];
  }

  if (fuseLocal_ && ctx_->size == 1) {
    // The whole step in one pass: every buffer := scale * reduce(all buffers).
    launchLocalAllreduceMany(ptrs_.data(), static_cast<int>(ptrs_.size()), count_, dt_, op_, static_cast<float>(scale_), *s0);
    noteLaunch();
  } else if (fuseLocal_) {
    // One launch: fold, exchange and fan-out inside the collective kernel.
    allreduce(*pc_, *reg_, regOffset_, count_, dt_, op_, algo_, *s0, ep);
  } else {
    // 1. fold the local pointers into ptrs_[0]
    if (multi) {
      std::vector<const void*> srcs(ptrs_.begin(), ptrs_.end());
      launchLocalReduceMany(ptrs_[0], srcs.data(), static_cast<int>(srcs.size()), count_, dt_, op_, *s0);
      noteLaunch();
    }
    // 2. across ranks
    if (ctx_->size > 1) {
      if (pc_ && literal_) {
        const size_t vecs = bytes / 16 / ctx_->size;
        int cap = shapeBlocks_ > 0 ? shapeBlocks_ : tuning().maxBlocks;
        if (const TuneEntry* e = TuningTable::get().lookup("allreduce_literal", ctx_->size, BufKind::REGISTERED, bytes)) {
          if (e->blocks > 0 && shapeBlocks_ == 0) cap = e->blocks;
        }
        const int blocks = std::max(1, std::min<int>({pc_->maxBlocks(), cap, static_cast<int>(vecs / kThreads) + 1}));
        pc_->checkHealth();
        pc_->orderStreams(*s0);
        pc_->launchGuard();
        launchSchedule(pc_->comm(), reg_->ptrsAt(regOffset_), pc_->stagePtrs(pc_->stageBytes() / 2), literal_->deviceTable,
                       static_cast<int>(literal_->schedule.steps.size()), scheduleBarriers(literal_->schedule), dt_, op_,
                       static_cast<float>(scale_), count_, reg_->vectorOk && regOffset_ % 16 == 0, blocks, *s0);
        noteLaunch();
        cudaError_t le = cudaGetLastError();
        if (le != cudaSuccess) GLB_THROW(Exception, "schedule kernel launch failed: ", cudaGetErrorString(le));
        pc_->markLaunched(*s0);
      } else if (pc_) {
        allreduce(*pc_, *reg_, regOffset_, count_, dt_, op_, algo_, *s0, ep);
      } else {
        runHostWorkspace(s0);
      }
    } else if (scale_ != 1.0) {
      void* one[1] = {ptrs_[0]};
      launchLocalAllreduceMany(one, 1, count_, dt_, op_, static_cast<float>(scale_), *s0);
      noteLaunch();
    }
    // 3. replicate to the other local pointers
    if (multi) {
      std::vector<void*> dsts(ptrs_.begin() + 1, ptrs_.end());
      launchLocalBroadcast(dsts.data(), static_cast<int>(dsts.size()), ptrs_[0], bytes, *s0);
      noteLaunch();
    }
  }

  if (multi) {
    s0.record();
    for (size_t i = 1; i < streams_.size(); i++) streams_[i].waitOn(s0);
  }
  if (syncOutputs_) {
    s0.record();
    s0.wait();
    if (pc_) pc_->checkHealth();
  }
}

// ---- broadcast --------------------------------------------------------------------------------

CudaBroadcastCore::CudaBroadcastCore(std::shared_ptr<Context> ctx, std::vector<void*> ptrs, size_t count,
                                     DataType dt, int rootRank, int rootPointerRank,
                                     std::vector<cudaStream_t> streams, Workspace ws)
    : ctx_(std::move(ctx)),
      ptrs_(std::move(ptrs)),
      count_(count),
      dt_(dt),
      root_(rootRank),
      rootPtr_(rootPointerRank),
      syncOutputs_(streams.empty()) {
  GLB_ENFORCE(!ptrs_.empty(), "need at least one pointer");
  GLB_ENFORCE(root_ >= 0 && root_ < ctx_->size, "invalid root rank ", root_);
  GLB_ENFORCE(rootPtr_ >= 0 && rootPtr_ < static_cast<int>(ptrs_.size()), "invalid root pointer rank");
  streams_ = makeStreams(ptrs_, streams);
  // The pointer that takes part in the cross-rank exchange: the root's source
  // pointer on the root, ptrs[0] elsewhere.
  const int idx = ctx_->rank == root_ ? rootPtr_ : 0;
  if (ctx_->size > 1 && peerPathUsable(ctx_, ws)) {
    auto pc = peerContextFor(ctx_, streams_[idx].getDeviceID());
    if (pc->peerAccessEverywhere()) {
      pc_ = pc;
      reg_ = pc_->resolveBuffer(ptrs_[idx], count_ * elementSize(dt_), &regOffset_);
    }
  }
  if (ctx_->size > 1 && !pc_) {
    GLB_CUDA_CHECK(cudaMallocHost(&hostScratch_, std::max<size_t>(count_ * elementSize(dt_), 16)));
  }
}

CudaBroadcastCore::~CudaBroadcastCore() {
  if (hostScratch_ != nullptr) cudaFreeHost(hostScratch_);
}

void CudaBroadcastCore::run() {
  if (count_ == 0) return;
  GLB_TRACE_RANGE("glb::CudaBroadcastOneToAll::run");
  const size_t bytes = count_ * elementSize(dt_);
  const bool isRoot = ctx_->rank == root_;
  const int idx = isRoot ? rootPtr_ : 0;
  CudaStream& s = streams_[idx];
  DeviceGuard g(s.getDeviceID());
  if (ctx_->size > 1) {
    if (pc_) {
      broadcast(*pc_, *reg_, regOffset_, bytes, root_, *s);
    } else {
      if (isRoot) {
        s.copyAsync(hostScratch_, ptrs_[idx], bytes);
        s.wait();
      }
      BroadcastOptions opts(ctx_);
      opts.setOutputRaw(hostScratch_, bytes);
      opts.setRoot(root_);
      opts.setTag(0x00CDA001u);
      glb::broadcast(opts);
      if (!isRoot) s.copyAsync(ptrs_[idx], hostScratch_, bytes);
    }
  }
  // Local fan-out to the remaining pointers.
  if (ptrs_.size() > 1) {
    std::vector<void*> dsts;
    for (size_t i = 0; i < ptrs_.size(); i++) {
      if (static_cast<int>(i) != idx) dsts.push_back(ptrs_[i]);
    }
    for (size_t i = 0; i < streams_.size(); i++) {
      if (static_cast<int>(i) == idx) continue;
      streams_[i].record();
      s.waitOn(streams_[i]);
    }
    launchLocalBroadcast(dsts.data(), static_cast<int>(dsts.size()), ptrs_[idx], bytes, *s);
    s.record();
    for (size_t i = 0; i < streams_.size(); i++) {
      if (static_cast<int>(i) != idx) streams_[i].waitOn(s);
    }
  }
  if (syncOutputs_) {
    s.record();
    s.wait();
  }
}

}  // namespace cuda

// ---- local allreduce -----------------------------------------------------------------------

template <typename T>
CudaAllreduceLocal<T>::CudaAllreduceLocal(const std::shared_ptr<Context>& context, const std::vector<T*>& ptrs,
                                          const size_t count, const std::vector<cudaStream_t>& streams)
    : Algorithm(context), ptrs_(cuda::eraseType(ptrs)), count_(count), syncOutputs_(streams.empty()) {
  streams_ = cuda::makeStreamsFor(ptrs_, streams);
}

template <typename T>
void CudaAllreduceLocal<T>::run() {
  if (count_ == 0 || ptrs_.size() < 2) return;
  cuda::CudaStream& s0 = streams_[0];
  cuda::DeviceGuard g(s0.getDeviceID());
  for (size_t i = 1; i < streams_.size(); i++) {
    streams_[i].record();
    s0.waitOn(streams_[i]);
  }
  // One pass: every buffer := sum of all buffers (peer buffers of other local GPUs are
  // read and written through peer access).
  cuda::launchLocalAllreduceMany(ptrs_.data(), static_cast<int>(ptrs_.size()), count_, DataTypeOf<T>::value, ReduceOp::SUM,
                                 1.0f, *s0);
  cuda::noteLaunch();
  s0.record();
  for (size_t i = 1; i < streams_.size(); i++) streams_[i].waitOn(s0);
  if (syncOutputs_) s0.wait();
}

template <typename T>
void CudaReductionFunction<T>::call(T* dst, const T* src, size_t n, cudaStream_t stream) const {
  cuda::launchLocalReduce(dst, src, n, DataTypeOf<T>::value, type_, stream);
}

#define GLB_INSTANTIATE(T)                    \
  template class CudaAllreduceLocal<T>;       \
  template class CudaReductionFunction<T>;
GLB_INSTANTIATE(int8_t)
GLB_INSTANTIATE(uint8_t)
GLB_INSTANTIATE(int32_t)
GLB_INSTANTIATE(int64_t)
GLB_INSTANTIATE(uint64_t)
GLB_INSTANTIATE(float)
GLB_INSTANTIATE(double)
GLB_INSTANTIATE(float16)
GLB_INSTANTIATE(bfloat16)
#undef GLB_INSTANTIATE

}  // namespace glb
