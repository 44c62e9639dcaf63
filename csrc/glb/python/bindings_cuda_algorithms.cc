// Old-style CUDA algorithm objects + remaining CUDA collectives for Python.
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include "glb/cuda/algorithms.h"
#include "glb/cuda/collectives.h"
#include "glb/cuda/nccl_wrapper.h"
#include "glb/cuda/schedules.h"

namespace py = pybind11;
using namespace glb;
using namespace glb::cuda;

namespace glb_py {

namespace {
inline void* P(uintptr_t p) { return reinterpret_cast<void*>(p); }
inline cudaStream_t S(uintptr_t s) { return reinterpret_cast<cudaStream_t>(s); }
std::vector<void*> ptrs(const std::vector<uintptr_t>& v) {
  std::vector<void*> o;
  for (auto p : v) o.push_back(P(p));
  return o;
}
std::vector<cudaStream_t> streams(const std::vector<uintptr_t>& v) {
  std::vector<cudaStream_t> o;
  for (auto s : v) o.push_back(S(s));
  return o;
}
}  // namespace

void registerCudaAlgorithms(py::module_& m) {
  py::class_<CudaAllreduceCore>(m, "CudaAllreduce")
      .def(py::init([](std::shared_ptr<Context> ctx, std::vector<uintptr_t> p, size_t count, int dtype, int op,
                       std::vector<uintptr_t> st, int algo, bool hostWorkspace) {
        py::gil_scoped_release nogil;
        return std::make_unique<CudaAllreduceCore>(std::move(ctx), ptrs(p), count, static_cast<DataType>(dtype),
                                                   static_cast<ReduceOp>(op), streams(st),
                                                   static_cast<AllreduceAlgo>(algo),
                                                   hostWorkspace ? Workspace::HOST : Workspace::PEER);
      }), py::arg("ctx"), py::arg("ptrs"), py::arg("count"), py::arg("dtype"), py::arg("op") = 1,
          py::arg("streams") = std::vector<uintptr_t>(), py::arg("algo") = 0, py::arg("host_workspace") = false)
      .def("run", [](CudaAllreduceCore& c) { py::gil_scoped_release nogil; c.run(); })
      .def("resolved_algo", [](CudaAllreduceCore& c) { return std::string(allreduceAlgoName(c.resolvedAlgo())); })
      .def("uses_peer_memory", &CudaAllreduceCore::usesPeerMemory)
      .def("set_scale", &CudaAllreduceCore::setScale, "Fused epilogue: result *= scale inside the collective kernel.")
      .def("set_launch_shape", &CudaAllreduceCore::setLaunchShape, py::arg("blocks") = 0, py::arg("unroll") = 0,
           py::arg("tile") = 0)
      .def("launches_per_run", &CudaAllreduceCore::launchesPerRun);

  py::class_<CudaBroadcastCore>(m, "CudaBroadcast")
      .def(py::init([](std::shared_ptr<Context> ctx, std::vector<uintptr_t> p, size_t count, int dtype, int root,
                       int rootPtr, std::vector<uintptr_t> st, bool hostWorkspace) {
        py::gil_scoped_release nogil;
        return std::make_unique<CudaBroadcastCore>(std::move(ctx), ptrs(p), count, static_cast<DataType>(dtype), root,
                                                   rootPtr, streams(st),
                                                   hostWorkspace ? Workspace::HOST : Workspace::PEER);
      }), py::arg("ctx"), py::arg("ptrs"), py::arg("count"), py::arg("dtype"), py::arg("root") = 0,
          py::arg("root_pointer") = 0, py::arg("streams") = std::vector<uintptr_t>(), py::arg("host_workspace") = false)
      .def("run", [](CudaBroadcastCore& c) { py::gil_scoped_release nogil; c.run(); });

  // NCCL comparator (baseline only).
  m.def("nccl_available", &ncclAvailable);
  m.def("nccl_version", &ncclVersionString);
  py::class_<NcclComm, std::shared_ptr<NcclComm>>(m, "NcclComm")
      .def_static("init_rank", [](std::shared_ptr<Context> ctx, int device) {
        py::gil_scoped_release nogil;
        return NcclComm::initRank(ctx, device);
      })
      .def_static("init_all", [](std::vector<int> devices) {
        py::gil_scoped_release nogil;
        return NcclComm::initAll(devices);
      })
      .def_property_readonly("rank", &NcclComm::rank)
      .def_property_readonly("size", &NcclComm::size)
      .def("allreduce", [](NcclComm& c, uintptr_t src, uintptr_t dst, size_t n, int dt, int op, uintptr_t st) {
        c.allreduce(P(src), P(dst), n, static_cast<DataType>(dt), static_cast<ReduceOp>(op), S(st));
      })
      .def("reduce", [](NcclComm& c, uintptr_t src, uintptr_t dst, size_t n, int dt, int op, int root, uintptr_t st) {
        c.reduce(P(src), P(dst), n, static_cast<DataType>(dt), static_cast<ReduceOp>(op), root, S(st));
      })
      .def("reduce_scatter", [](NcclComm& c, uintptr_t src, uintptr_t dst, size_t n, int dt, int op, uintptr_t st) {
        c.reduceScatter(P(src), P(dst), n, static_cast<DataType>(dt), static_cast<ReduceOp>(op), S(st));
      })
      .def("broadcast", [](NcclComm& c, uintptr_t src, uintptr_t dst, size_t n, int dt, int root, uintptr_t st) {
        c.broadcast(P(src), P(dst), n, static_cast<DataType>(dt), root, S(st));
      })
      .def("allgather", [](NcclComm& c, uintptr_t src, uintptr_t dst, size_t n, int dt, uintptr_t st) {
        c.allgather(P(src), P(dst), n, static_cast<DataType>(dt), S(st));
      })
      .def("alltoall", [](NcclComm& c, uintptr_t src, uintptr_t dst, size_t n, int dt, uintptr_t st) {
        c.alltoall(P(src), P(dst), n, static_cast<DataType>(dt), S(st));
      })
      .def("sendrecv", [](NcclComm& c, uintptr_t src, int dst, uintptr_t dstBuf, int srcRank, size_t n, int dt, uintptr_t st) {
        c.sendrecv(P(src), dst, P(dstBuf), srcRank, n, static_cast<DataType>(dt), S(st));
      })
      .def("mem_alloc", [](NcclComm& c, size_t bytes) { return reinterpret_cast<uintptr_t>(c.memAlloc(bytes)); },
           "ncclMemAlloc: a buffer NCCL can register for NVLS / zero-copy.")
      .def("mem_free", [](NcclComm& c, uintptr_t p) { c.memFree(P(p)); })
      .def("register_buffer", [](NcclComm& c, uintptr_t p, size_t bytes) {
        return reinterpret_cast<uintptr_t>(c.registerBuffer(P(p), bytes));
      })
      .def("deregister_buffer", [](NcclComm& c, uintptr_t h) { c.deregisterBuffer(P(h)); });

  // Step tables of the literal schedules (pure host code: testable without a GPU).
  m.def("build_schedule", [](const std::string& name, int rank, int size, size_t count, int base, size_t pack) {
    Schedule sc;
    if (name == "ring") sc = buildRingSchedule(rank, size, count, pack);
    else if (name == "ring_chunked") sc = buildRingChunkedSchedule(rank, size, count, pack);
    else if (name == "halving_doubling") sc = buildHalvingDoublingSchedule(rank, size, count, pack);
    else if (name == "halving_doubling_pipelined") sc = buildHalvingDoublingPipelinedSchedule(rank, size, count, pack, base);
    else if (name == "bcube") sc = buildBcubeSchedule(rank, size, count, base, pack);
    else GLB_THROW_INVALID_OPERATION_EXCEPTION("unknown schedule ", name);
    py::list out;
    for (const auto& st : sc.steps) {
      py::dict d;
      d["mode"] = st.mode;
      d["from_stage"] = st.fromStage;
      d["off"] = st.off;
      d["len"] = st.len;
      d["sync"] = st.sync;
      py::list peers;
      for (int i = 0; i < st.npeers; i++) peers.append(st.peers[i]);
      d["peers"] = peers;
      out.append(d);
    }
    return out;
  }, py::arg("name"), py::arg("rank"), py::arg("size"), py::arg("count"), py::arg("base") = 2, py::arg("pack") = 4);

  m.def("peer_context_for", [](std::shared_ptr<Context> ctx, int device, size_t stageBytes, bool useVmm, bool useNvls) {
    PeerOptions o;
    if (stageBytes > 0) o.stageBytes = stageBytes;
    o.useVmm = useVmm;
    o.useNvls = useNvls;
    py::gil_scoped_release nogil;
    return peerContextFor(ctx, device, o);
  }, py::arg("ctx"), py::arg("device"), py::arg("stage_bytes") = 0, py::arg("use_vmm") = true, py::arg("use_nvls") = true,
     "The PeerContext attached to (ctx, device); created collectively on first use with the given options.");
  m.def("release_peer_contexts", [](std::shared_ptr<Context> ctx) { releasePeerContexts(ctx); });

  // ---- data movement: registered (`*_reg`) and staged (plain pointer) flavours ------------
  m.def("broadcast_reg", [](PeerContext& pc, const PeerBuffer& b, size_t off, size_t bytes, int root, uintptr_t st) {
    py::gil_scoped_release nogil;
    broadcast(pc, b, off, bytes, root, S(st));
  });
  m.def("broadcast", [](PeerContext& pc, uintptr_t p, size_t bytes, int root, uintptr_t st) {
    py::gil_scoped_release nogil;
    broadcast(pc, P(p), bytes, root, S(st));
  });
  m.def("allgatherv_reg", [](PeerContext& pc, uintptr_t in, const PeerBuffer& out, size_t off,
                             std::vector<size_t> bytesPerRank, uintptr_t st) {
    py::gil_scoped_release nogil;
    allgatherv(pc, P(in), out, off, bytesPerRank, S(st));
  });
  m.def("allgatherv", [](PeerContext& pc, uintptr_t in, uintptr_t out, std::vector<size_t> bytesPerRank, uintptr_t st) {
    py::gil_scoped_release nogil;
    allgatherv(pc, P(in), P(out), bytesPerRank, S(st));
  });
  m.def("gatherv_reg", [](PeerContext& pc, uintptr_t in, const PeerBuffer& out, size_t off,
                          std::vector<size_t> bytesPerRank, int root, uintptr_t st) {
    py::gil_scoped_release nogil;
    gatherv(pc, P(in), out, off, bytesPerRank, root, S(st));
  });
  m.def("gatherv", [](PeerContext& pc, uintptr_t in, uintptr_t out, std::vector<size_t> bytesPerRank, int root,
                      uintptr_t st) {
    py::gil_scoped_release nogil;
    gatherv(pc, P(in), P(out), bytesPerRank, root, S(st));
  });
  m.def("alltoallv_reg", [](PeerContext& pc, uintptr_t in, std::vector<size_t> sendBytes, const PeerBuffer& out,
                            size_t off, std::vector<size_t> recvBytes, uintptr_t st) {
    py::gil_scoped_release nogil;
    alltoallv(pc, P(in), sendBytes, out, off, recvBytes, S(st));
  });
  m.def("alltoallv", [](PeerContext& pc, uintptr_t in, std::vector<size_t> sendBytes, uintptr_t out,
                        std::vector<size_t> recvBytes, uintptr_t st) {
    py::gil_scoped_release nogil;
    alltoallv(pc, P(in), sendBytes, P(out), recvBytes, S(st));
  });
  m.def("alltoall_reg", [](PeerContext& pc, uintptr_t in, const PeerBuffer& out, size_t off, size_t bytes, uintptr_t st) {
    py::gil_scoped_release nogil;
    alltoall(pc, P(in), out, off, bytes, S(st));
  });
  m.def("alltoall", [](PeerContext& pc, uintptr_t in, uintptr_t out, size_t bytes, uintptr_t st) {
    py::gil_scoped_release nogil;
    alltoall(pc, P(in), P(out), bytes, S(st));
  });
  m.def("scatter_reg", [](PeerContext& pc, uintptr_t in, const PeerBuffer& out, size_t off, size_t bytes, int root,
                          uintptr_t st) {
    py::gil_scoped_release nogil;
    scatter(pc, P(in), out, off, bytes, root, S(st));
  });
  m.def("scatter", [](PeerContext& pc, uintptr_t in, uintptr_t out, size_t bytes, int root, uintptr_t st) {
    py::gil_scoped_release nogil;
    scatter(pc, P(in), P(out), bytes, root, S(st));
  });
  m.def("reduce_scatter_reg", [](PeerContext& pc, const PeerBuffer& in, size_t off, uintptr_t out,
                                 std::vector<size_t> counts, int dtype, int op, uintptr_t st, double scale) {
    py::gil_scoped_release nogil;
    reduce_scatter(pc, in, off, P(out), counts, static_cast<DataType>(dtype), static_cast<ReduceOp>(op), S(st), scale);
  }, py::arg("pc"), py::arg("input"), py::arg("offset"), py::arg("output"), py::arg("counts"), py::arg("dtype"),
     py::arg("op") = 1, py::arg("stream") = 0, py::arg("scale") = 1.0);
  m.def("reduce_scatter", [](PeerContext& pc, uintptr_t in, uintptr_t out, std::vector<size_t> counts, int dtype,
                             int op, uintptr_t st, double scale) {
    py::gil_scoped_release nogil;
    reduce_scatter(pc, P(in), P(out), counts, static_cast<DataType>(dtype), static_cast<ReduceOp>(op), S(st), scale);
  }, py::arg("pc"), py::arg("input"), py::arg("output"), py::arg("counts"), py::arg("dtype"), py::arg("op") = 1,
     py::arg("stream") = 0, py::arg("scale") = 1.0);
  // With a dtype conversion (f32 <-> f16 / bf16). Counts are ELEMENTS: input and output
  // element sizes differ.
  m.def("reduce_scatter_cast_reg", [](PeerContext& pc, const PeerBuffer& in, size_t off, uintptr_t out,
                                      std::vector<size_t> counts, int dtype, int outDtype, int op, uintptr_t st,
                                      double scale) {
    py::gil_scoped_release nogil;
    reduceScatterCast(pc, in, off, P(out), counts, static_cast<DataType>(dtype), static_cast<DataType>(outDtype),
                      static_cast<ReduceOp>(op), S(st), scale);
  }, py::arg("pc"), py::arg("input"), py::arg("offset"), py::arg("output"), py::arg("counts"), py::arg("dtype"),
     py::arg("out_dtype"), py::arg("op") = 1, py::arg("stream") = 0, py::arg("scale") = 1.0);
  m.def("reduce_scatter_cast", [](PeerContext& pc, uintptr_t in, uintptr_t out, std::vector<size_t> counts, int dtype,
                                  int outDtype, int op, uintptr_t st, double scale) {
    py::gil_scoped_release nogil;
    reduceScatterCast(pc, P(in), P(out), counts, static_cast<DataType>(dtype), static_cast<DataType>(outDtype),
                      static_cast<ReduceOp>(op), S(st), scale);
  }, py::arg("pc"), py::arg("input"), py::arg("output"), py::arg("counts"), py::arg("dtype"), py::arg("out_dtype"),
     py::arg("op") = 1, py::arg("stream") = 0, py::arg("scale") = 1.0);
  m.def("allgatherv_cast_reg", [](PeerContext& pc, uintptr_t in, int dtype, const PeerBuffer& out, size_t off,
                                  std::vector<size_t> counts, int outDtype, uintptr_t st) {
    py::gil_scoped_release nogil;
    allgathervCast(pc, P(in), static_cast<DataType>(dtype), out, off, counts, static_cast<DataType>(outDtype), S(st));
  });
  m.def("allgatherv_cast", [](PeerContext& pc, uintptr_t in, int dtype, uintptr_t out, std::vector<size_t> counts,
                              int outDtype, uintptr_t st) {
    py::gil_scoped_release nogil;
    allgathervCast(pc, P(in), static_cast<DataType>(dtype), P(out), counts, static_cast<DataType>(outDtype), S(st));
  });
  m.def("reduce_reg", [](PeerContext& pc, const PeerBuffer& in, size_t inOff, const PeerBuffer& out, size_t outOff,
                         size_t count, int dtype, int op, int root, uintptr_t st) {
    py::gil_scoped_release nogil;
    reduce(pc, in, inOff, out, outOff, count, static_cast<DataType>(dtype), static_cast<ReduceOp>(op), root, S(st));
  });
  m.def("reduce", [](PeerContext& pc, uintptr_t in, uintptr_t out, size_t count, int dtype, int op, int root,
                     uintptr_t st) {
    py::gil_scoped_release nogil;
    reduce(pc, P(in), P(out), count, static_cast<DataType>(dtype), static_cast<ReduceOp>(op), root, S(st));
  });
}

}  // namespace glb_py
