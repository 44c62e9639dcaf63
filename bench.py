#!/usr/bin/env python
"""Headline benchmark: cuda_allreduce_ring_chunked, float32, on N B200s of one node.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python bench.py --gpus 1 --steps 20 --warmup 5 --dump-outputs DIR   # + the last step's buffers as DIR/*.npy
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29500 bench.py --gpus 8 --steps 20 --warmup 5
    ... bench.py --impl reference ...   # unmodified pytorch/gloo benchmark_cuda from baseline/_ref

A *step* is one `CudaAllreduceRingChunked.run()` on a 1e8-element float32 buffer per
GPU (400 MB, larger than the 126 MB L2, so back-to-back steps cannot hit in cache).
Timing: CUDA events on the launching stream around exactly K steps, barrier +
synchronize on both sides, max over ranks. `value` is the allreduce bus bandwidth
(algbw * 2(N-1)/N, GB/s per GPU — the figure BASELINE.json asks for, against the
900 GB/s/direction NVLink roofline). With N=1 a one-buffer allreduce is the
identity, so the N=1 run uses two local buffers per rank (`--inputs 2`, which the
reference's benchmark supports too) and reports algorithm bandwidth instead.
The JSON also carries a latency sweep (p50/p99, L2 flushed between iterations),
an end-to-end number (pinned-host H2D of the input and D2H of the result every
step) and the clocks seen while timing.
"""
from __future__ import annotations

import argparse
import glob
import json
import os
import re
import shutil
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# `value` is the whole-job aggregate the driver contract asks for: the per-GPU bus bandwidth
# (algbw x 2(N-1)/N, the number NCCL-style tables quote and `busbw_gbs` keeps) summed over the
# N GPUs. At N=1 there is no bus: the step is the local reduce + re-broadcast of the two
# buffers and the value is its algorithm bandwidth.
METRIC = ("cuda_allreduce_ring_chunked float32 aggregate bus bandwidth (GB/s summed over the N GPUs = "
          "N x algbw x 2(N-1)/N; algbw at N=1)")
PUBLISHED_BUSBW_GBS = 2.8  # BASELINE.md: 20 MB allreduce_ring_chunked, 4 machines, 40 GbE (derived busbw)
HEADLINE_ELEMENTS = 100_000_000
SWEEP = [1, 10, 100, 1_000, 10_000, 100_000, 1_000_000, 10_000_000]
DUMP_BYTES = 32 << 20  # --dump-outputs budget over all ranks; larger outputs are sampled down to it
DUMP_SEED = 0


def env_int(name, dflt):
    return int(os.environ.get(name, dflt))


def rendezvous_dir(tag: str) -> str:
    port = os.environ.get("MASTER_PORT", "0")
    launcher = os.getppid() if "RANK" in os.environ else os.getpid()
    return f"/tmp/glb_bench_{tag}_{port}_{launcher}"


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(out_dir, tensors, rank, world):
    """Writes the buffers a step hands back to its caller as <out_dir>/rank<r>_buffer<i>.npy (float32).
    A buffer larger than its share of DUMP_BYTES is cut into that many equal slices and reduced to
    one value per slice, at a position drawn from DUMP_SEED: the same positions on every run, so two
    builds compare element for element."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    per = DUMP_BYTES // 4 // (world * len(tensors))
    for i, t in enumerate(tensors):
        n = t.numel()
        if n > per:
            lo = np.arange(per, dtype=np.int64) * n // per
            hi = np.append(lo[1:], n)
            idx = np.random.default_rng(DUMP_SEED).integers(lo, hi)
            t = t.index_select(0, torch.from_numpy(idx).to(t.device))
        np.save(os.path.join(out_dir, f"rank{rank}_buffer{i}.npy"), t.float().cpu().numpy())


# ------------------------------------------------------------------------------------------
# our implementation
# ------------------------------------------------------------------------------------------

MOVE_SIZES = [1 << 10, 8 << 10, 64 << 10, 512 << 10, 4 << 20, 32 << 20, 256 << 20, 1 << 30]  # bytes per rank buffer
HALF_ELEMENTS = [100_000, 10_000_000, 100_000_000]  # fp16 halving-doubling / bcube (BASELINE config 3)


def run_ours(args):
    import numpy as np
    import torch

    import gloo_b200 as gb
    from gloo_b200.ops import cuda as gcu

    rank, world = env_int("RANK", 0), env_int("WORLD_SIZE", 1)
    local = env_int("LOCAL_RANK", 0)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # Keep this rank (its pinned staging buffers and the transport's I/O thread) on the
    # socket its GPU hangs off.
    from gloo_b200.utils.affinity import bind_to_gpu
    cpus = bind_to_gpu(local)
    cu = gb._C.cuda

    store = gb.FileStore(rendezvous_dir("ours"))
    ctx = gb.init_context(rank, world, store=store, device=gb.create_device("127.0.0.1"), timeout_ms=120000)
    inputs = 2 if world == 1 else 1
    cc = gcu.CudaContext(ctx, local, stage_bytes=256 << 20)
    stream = torch.cuda.Stream()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > L2
    F32, F16, U8 = int(gb.DataType.FLOAT32), int(gb.DataType.FLOAT16), int(gb.DataType.UINT8)
    bus = (lambda algbw: algbw * 2 * (world - 1) / world) if world > 1 else (lambda algbw: None)

    def host_max(values):
        arr = np.asarray(values, dtype=np.float64).copy()
        if world > 1:
            gb.allreduce(ctx, arr, op=gb.ReduceOp.MAX)
        return arr

    def sync_all():
        torch.cuda.synchronize()
        gb.barrier(ctx)

    def time_k(fn, k=None, warm=3):
        """K back-to-back calls, device timed on the launching stream, max over ranks -> ms per call."""
        k = k or args.steps
        for _ in range(warm):
            fn()
        sync_all()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(k):
            fn()
        b.record(stream)
        stream.synchronize()
        sync_all()
        return float(host_max([a.elapsed_time(b)])[0]) / k

    def latency(fn, iters, nbytes):
        """Per-call events with the L2 flushed in between; the whole batch is queued behind a
        5 ms spin so that host jitter cannot starve the GPU queue. -> (p50, p99, min) in us."""
        with torch.cuda.stream(stream):
            for _ in range(max(3, args.warmup)):  # dry batch under the same conditions (flushed L2)
                if nbytes < (128 << 20):
                    flush.fill_(0)
                fn()
        sync_all()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        with torch.cuda.stream(stream):
            cu.spin(8_000_000, stream.cuda_stream)
            for a, b in evs:
                if nbytes < (128 << 20):
                    flush.fill_(0)
                a.record(stream)
                fn()
                b.record(stream)
        stream.synchronize()
        sync_all()
        per = host_max([a.elapsed_time(b) * 1e3 for a, b in evs])
        per.sort()
        return float(per[len(per) // 2]), float(per[min(len(per) - 1, int(len(per) * 0.99))]), float(per[0])

    def verify_full(t, start, stride, rtol=1e-5, atol=0.0, what=""):
        """Whole buffer, every rank, on the device (closed form in fp64)."""
        code = {torch.float32: F32, torch.float16: F16, torch.bfloat16: int(gb.DataType.BFLOAT16)}[t.dtype]
        bad, first = cu.verify(t.data_ptr(), t.numel(), code, float(start), float(stride), rtol, atol, stream.cuda_stream)
        worst = int(host_max([bad])[0])
        if worst:
            raise AssertionError(f"verification failed ({what}): {bad} wrong elements on rank {rank}, first at {first}")

    def fill(t, start, stride):
        code = {torch.float32: F32, torch.float16: F16, torch.bfloat16: int(gb.DataType.BFLOAT16)}[t.dtype]
        cu.fill(t.data_ptr(), t.numel(), code, float(start), float(stride), stream.cuda_stream)

    # ---- correctness matrix on the real multi-GPU path (before anything is timed) ---------------
    verified = {}
    if world > 1 and not args.no_verify_matrix:
        tri = world * (world - 1) / 2
        with torch.cuda.stream(stream):
            for dtype, tol in ((torch.float32, 1e-6), (torch.float16, 2e-3), (torch.bfloat16, 1.6e-2)):
                for n in (1000, 1 << 20, 5_000_001):
                    mod_ok = dtype == torch.float32
                    for kind in ("sym", "reg", "user"):
                        algos = ["auto"]
                        if kind != "user":
                            algos.append("two_shot")
                        if kind == "sym" and cc.nvls_available():
                            algos.append("nvls")
                            if world in (2, 4, 8) and n > 1000:
                                algos.append("hybrid")
                        if kind == "user" and n > 1000:
                            algos.append("pipelined")
                        if n * 4 <= 32768:
                            algos += ["ll", "one_shot"]
                        t = cc.empty(n, dtype) if kind == "sym" else torch.empty(n, dtype=dtype, device=dev)
                        if kind == "reg":
                            cc.register(t)
                        for algo in algos:
                            # values stay exactly representable: start = rank (x 1/64 for 16-bit), stride 0 or 1
                            if mod_ok:
                                fill(t, rank, world)
                                cc.allreduce(t, algo=algo, stream=stream)
                                verify_full(t, tri, world * world, tol, 0.0, f"allreduce {dtype} {kind} {algo} {n}")
                            else:
                                fill(t, (rank + 1) / 64.0, 0.0)
                                cc.allreduce(t, algo=algo, stream=stream, average=True)
                                verify_full(t, (tri + world) / 64.0 / world, 0.0, tol, 1e-3, f"allreduce {dtype} {kind} {algo} {n}")
                            verified[f"allreduce_{str(dtype).split('.')[-1]}_{kind}_{algo}"] = True
                        del t
            # fused cast epilogue, data movement, point to point
            n = 1 << 20
            a32, o16 = cc.empty(n, torch.float32), cc.empty(n, torch.bfloat16)
            fill(a32, rank + 1, 0.0)
            cc.allreduce(a32, out=o16, stream=stream, average=True)
            verify_full(o16, (tri + world) / world, 0.0, 1e-2, 0.0, "cast epilogue")
            verified["allreduce_cast_f32_to_bf16_avg"] = True
            per = 250_003
            out = torch.zeros(per * world, device=dev)
            cc.allgather(out, torch.full((per,), float(rank), device=dev), stream=stream)
            a_in = torch.cat([torch.full((per,), float(rank * 100 + j), device=dev) for j in range(world)])
            a_out = torch.zeros(per * world, device=dev)
            cc.alltoall(a_out, a_in, stream=stream)
            counts = [1000 * (j + 1) + 1 for j in range(world)]
            send = [counts[(rank + j) % world] for j in range(world)]  # uneven, 4-byte aligned offsets
            recv = [counts[(j + rank) % world] for j in range(world)]
            # rank r sends counts[(r+j)%P] to j; rank j receives from r counts[(r+j)%P] = its recv[r]
            v_in = torch.cat([torch.full((send[j],), float(rank * 100 + j), device=dev) for j in range(world)])
            v_out = torch.zeros(sum(recv), device=dev)
            cc.alltoallv(v_out, recv, v_in, send, stream=stream)
            rs_in = torch.empty(per * world, device=dev)
            fill(rs_in, rank, world)
            rs_out = torch.zeros(per, device=dev)
            cc.reduce_scatter(rs_out, rs_in, stream=stream)
            bc = cc.empty(1 << 20, torch.float32)
            fill(bc, rank, 1.0)
            cc.broadcast(bc, root=world - 1, stream=stream)
            nxt, prv = (rank + 1) % world, (rank - 1) % world
            s_t, r_t = torch.full((3_000_001,), float(rank), device=dev), torch.zeros(3_000_001, device=dev)
            cc.sendrecv(s_t, nxt, r_t, prv, stream=stream)
            # zero-copy exchange between two symmetric buffers; relay broadcast (forced: the table only picks it from 64 MB)
            xa, xb = cc.empty(3_000_001, torch.float32), cc.empty(3_000_001, torch.float32)
            xa.fill_(float(rank))
            xb.zero_()
        sync_all()
        with torch.cuda.stream(stream):
            cc.exchange(xa, nxt, xb, prv, stream=stream)
            rb = cc.empty(5_000_001, torch.float32)
            fill(rb, rank, 1.0)
            if world > 2:
                os.environ["GLB_CUDA_BCAST_MODE"] = "3"
            cc.broadcast(rb, root=1 % world, stream=stream)
            os.environ.pop("GLB_CUDA_BCAST_MODE", None)
        stream.synchronize()
        assert float(xb[0]) == prv and float(xb[-1]) == prv and float(xb[1_500_000]) == prv, "exchange"
        verify_full(rb, 1 % world, 1.0, 0.0, 0.0, "relay broadcast")
        verified["exchange"] = True
        verified["broadcast_relay" if world > 2 else "broadcast_root1"] = True
        exp_g = torch.arange(world, device=dev).repeat_interleave(per).float()
        assert torch.equal(out, exp_g), "allgather"
        assert torch.equal(a_out, torch.cat([torch.full((per,), float(j * 100 + rank), device=dev) for j in range(world)])), "alltoall"
        assert torch.equal(v_out, torch.cat([torch.full((recv[j],), float(j * 100 + rank), device=dev) for j in range(world)])), "alltoallv"
        verify_full(rs_out, rank * per * world * world + tri, world * world, 1e-6, 0.0, "reduce_scatter")
        verify_full(bc, world - 1, 1.0, 0.0, 0.0, "broadcast")
        assert float(r_t[0]) == prv and float(r_t[-1]) == prv, "sendrecv"
        for k in ("allgather", "alltoall", "alltoallv", "reduce_scatter", "broadcast", "sendrecv"):
            verified[k] = True
        cc.check_health()
        del a32, o16, out, a_in, a_out, v_in, v_out, rs_in, rs_out, bc, s_t, r_t, xa, xb, rb
        sync_all()

    def make(elements, symmetric=True, dtype=torch.float32, cls=None, literal=False):
        # The harness owns the buffers (as the reference's benchmark does). By default they
        # come from the library's symmetric allocator: peer-mapped and, on >2 GPUs, bound to
        # an NVSwitch multicast object so the reduction can run inside the switch. Plain
        # cudaMalloc'ed tensors (symmetric=False) are registered through cudaIpc instead.
        if symmetric:
            ts = [cc.empty(elements, dtype) for _ in range(inputs)]
        else:
            ts = [torch.empty(elements, dtype=dtype, device=dev) for _ in range(inputs)]
        algo = (cls or gcu.CudaAllreduceRingChunked)(ctx, ts, streams=[stream] * inputs, literal=literal)
        return ts, algo

    total = world * inputs
    tri_all = total * (total - 1) / 2

    def fill_inputs(ts):
        for i, t in enumerate(ts):
            fill(t, rank * inputs + i, total)

    def check_outputs(ts, what):
        for t in ts:
            verify_full(t, tri_all, total * total, 1e-5, 0.0, what)

    # ---- headline: K back-to-back steps, device timed ------------------------------------
    E = args.elements
    ts, algo = make(E)
    with torch.cuda.stream(stream):
        fill_inputs(ts)
        algo.run()
    check_outputs(ts, "headline, before timing")  # whole buffer, every rank
    for _ in range(args.warmup):
        algo.run()
    sync_all()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = cu.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    ev0.record(stream)
    for _ in range(args.steps):
        algo.run()
    ev1.record(stream)
    stream.synchronize()
    sync_all()
    launches = cu.launch_count() - launches0
    total_ms = float(host_max([ev0.elapsed_time(ev1)])[0])
    ms_per_step = total_ms / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ts, rank, world)
    with torch.cuda.stream(stream):
        fill_inputs(ts)
        algo.run()
    check_outputs(ts, "headline, after timing")
    cc.check_health()
    size_bytes = E * 4
    algbw = size_bytes / (ms_per_step * 1e-3) / 1e9
    busbw = bus(algbw)
    resolved = algo.resolved_algo() if world > 1 else "local_fused"
    plan = cc.plan(ts[0]) if world > 1 else {}

    # ---- end to end: pinned host -> device, allreduce, device -> pinned host, every step ----
    # The call a user with host-resident data makes: gcu.CudaHostAllreduce, which pipelines
    # the PCIe legs with the NVLink reduction piece by piece (same kernels as above).
    del ts, algo
    hins = [torch.empty(E, dtype=torch.float32).pin_memory() for _ in range(inputs)]
    for h in hins:
        h.fill_(1.0)
    hout = torch.empty(E, dtype=torch.float32).pin_memory()
    e2e = gcu.CudaHostAllreduce(ctx, cc, hins, hout, chunks=args.e2e_chunks)

    def e2e_step():
        with torch.cuda.stream(stream):
            e2e.run()
    e2e_ms = time_k(e2e_step, warm=min(3, args.warmup))
    # The sampler ran through both timed regions (device-only steps and end-to-end steps).
    clocks = sampler.stop() if rank == 0 else None
    assert abs(float(hout[0]) - world * inputs) < 1e-3 and abs(float(hout[-1]) - world * inputs) < 1e-3, "e2e result mismatch"
    e2e_algbw = size_bytes / (e2e_ms * 1e-3) / 1e9
    e2e_val = bus(e2e_algbw) if world > 1 else e2e_algbw
    e2e_launches = e2e.launches_per_run
    del hins, hout, e2e

    extra, configs = {}, {}
    nccl = None
    if world > 1:
        try:
            nccl = cu.NcclComm.init_rank(ctx, local)
        except Exception as e:  # noqa: BLE001
            extra["nccl_comparator"] = {"unavailable": str(e)[:200]}

    def busbw_of(nbytes, ms, factor):
        return round(nbytes / (ms * 1e-3) / 1e9 * factor, 3)

    ar_factor = 2 * (world - 1) / world if world > 1 else 1.0
    if world > 1 and not args.quick:
        # ---- the link: one-directional peer copy by our own put kernel (roofline denominator) -----
        win = cc.empty(64 << 20, torch.float32)
        src = torch.ones(64 << 20, device=dev)
        sync_all()
        put_ms = time_k(lambda: cc.put(src, win, (rank + 1) % world, stream=stream), k=10)
        peer_copy_gbs = round((256 << 20) / (put_ms * 1e-3) / 1e9, 1)
        cu.set_tuning({"tma_copies": True})   # the same copy through cp.async.bulk (TMA, one issuing thread per CTA)
        tma_ms = time_k(lambda: cc.put(src, win, (rank + 1) % world, stream=stream), k=10)
        cu.set_tuning({"tma_copies": False})
        extra["peer_copy_gbs_tma"] = round((256 << 20) / (tma_ms * 1e-3) / 1e9, 1)
        peer_copy_gbs = max(peer_copy_gbs, extra["peer_copy_gbs_tma"])
        del win, src
        # ---- same size on plain cudaMalloc'ed buffers: registered (cudaIpc) and unregistered ---------
        pts, palgo = make(E, symmetric=False)
        with torch.cuda.stream(stream):
            fill_inputs(pts)
            palgo.run()
        check_outputs(pts, "cudaIpc-registered buffers")
        pms = time_k(palgo.run)
        extra["plain_cudamalloc_buffers"] = {"ms_per_step": round(pms, 5), "variant": palgo.resolved_algo(),
                                             "busbw_gbs": busbw_of(size_bytes, pms, ar_factor),
                                             "note": "cudaMalloc'ed tensors registered through cudaIpc at construction"}
        del palgo
        with torch.cuda.stream(stream):
            fill_inputs(pts)
            cc.allreduce(pts[0], stream=stream)
        check_outputs(pts[:1], "unregistered pointer (pipelined)")
        ums = time_k(lambda: cc.allreduce(pts[0], stream=stream))
        extra["unregistered_pointer"] = {"ms_per_step": round(ums, 5), "variant": cc.plan(pts[0])["algo"],
                                         "busbw_gbs": busbw_of(size_bytes, ums, ar_factor),
                                         "note": "arbitrary T*: in-kernel copy-in / NVLS exchange / copy-out pipeline through the pool"}
        if nccl is not None:
            ptr = pts[0].data_ptr()
            nms = time_k(lambda: nccl.allreduce(ptr, ptr, E, F32, 1, stream.cuda_stream))
            comp = {"ms_per_step": round(nms, 5), "version": cu.nccl_version(), "busbw_gbs": busbw_of(size_bytes, nms, ar_factor),
                    "buffers": "plain cudaMalloc"}
            try:
                nb = nccl.mem_alloc(size_bytes)
                handle = nccl.register_buffer(nb, size_bytes)
                rms = time_k(lambda: nccl.allreduce(nb, nb, E, F32, 1, stream.cuda_stream))
                comp["registered"] = {"ms_per_step": round(rms, 5), "busbw_gbs": busbw_of(size_bytes, rms, ar_factor),
                                      "buffers": "ncclMemAlloc + ncclCommRegister (NCCL's zero-copy / NVLS user buffers)"}
                torch.cuda.synchronize()
                nccl.deregister_buffer(handle)
                nccl.mem_free(nb)
            except Exception as e:  # noqa: BLE001
                comp["registered"] = {"unavailable": str(e)[:200]}
            extra["nccl_comparator"] = comp
        del pts

        # ---- BASELINE config 3: fp16 halving-doubling / bcube classes ------------------------------------
        for name, cls in (("cuda_allreduce_halving_doubling_fp16", gcu.CudaAllreduceHalvingDoubling),
                          ("cuda_allreduce_bcube_fp16", gcu.CudaAllreduceBcube)):
            rows = []
            for n in HALF_ELEMENTS:
                row = {"elements": n, "bytes": n * 2}
                for literal in (False, True):
                    hts, halgo = make(n, dtype=torch.float16, cls=cls, literal=literal)
                    with torch.cuda.stream(stream):
                        fill(hts[0], (rank + 1) / 64.0, 0.0)
                        halgo.run()
                    verify_full(hts[0], (world * (world + 1) / 2) / 64.0, 0.0, 2e-3, 0.0, f"{name} literal={literal}")
                    ms = time_k(halgo.run, k=max(5, args.steps // 2))
                    key = "literal" if literal else "auto"
                    row[key] = {"ms": round(ms, 5), "busbw_gbs": busbw_of(n * 2, ms, ar_factor), "variant": halgo.resolved_algo()}
                    del hts, halgo
                if nccl is not None:
                    ht = torch.ones(n, dtype=torch.float16, device=dev)
                    ms = time_k(lambda: nccl.allreduce(ht.data_ptr(), ht.data_ptr(), n, F16, 1, stream.cuda_stream), k=max(5, args.steps // 2))
                    row["nccl"] = {"ms": round(ms, 5), "busbw_gbs": busbw_of(n * 2, ms, ar_factor)}
                    del ht
                rows.append(row)
            configs[name] = rows

        # ---- BASELINE configs 4 + 5: allgather / alltoall(v) / reduce_scatter / broadcast, 1 KB - 1 GB ----
        mv_factor = (world - 1) / world
        for coll in ("allgather", "alltoall", "alltoall_v", "reduce_scatter", "cuda_broadcast_one_to_all"):
            rows = []
            for nbytes in MOVE_SIZES:
                per = max(16, nbytes // world // 16 * 16)
                tot = per * world
                if coll == "cuda_broadcast_one_to_all":
                    tot = max(16, nbytes // 16 * 16)
                iters = 20 if tot <= (64 << 20) else 6
                ours_fn = nccl_fn = None
                if coll == "allgather":
                    o, i = cc.empty(tot, torch.uint8), torch.ones(per, dtype=torch.uint8, device=dev)
                    ours_fn = lambda: cc.allgather(o, i, stream=stream)  # noqa: E731
                    if nccl is not None:
                        nccl_fn = lambda: nccl.allgather(i.data_ptr(), o.data_ptr(), per, U8, stream.cuda_stream)  # noqa: E731
                elif coll == "alltoall":
                    o, i = cc.empty(tot, torch.uint8), torch.ones(tot, dtype=torch.uint8, device=dev)
                    ours_fn = lambda: cc.alltoall(o, i, stream=stream)  # noqa: E731
                    if nccl is not None:
                        nccl_fn = lambda: nccl.alltoall(i.data_ptr(), o.data_ptr(), per, U8, stream.cuda_stream)  # noqa: E731
                elif coll == "alltoall_v":
                    # uneven split (1 : 2 : ... : P) on offsets that are only 4-byte aligned
                    unit = max(4, tot // (world * (world + 1) // 2) // 4 * 4)
                    cnt = [unit * (j + 1) + 4 for j in range(world)]
                    send = [cnt[(rank + j) % world] for j in range(world)]
                    recv = [cnt[(j + rank) % world] for j in range(world)]
                    o = cc.empty(sum(recv), torch.uint8)
                    i = torch.ones(sum(send), dtype=torch.uint8, device=dev)
                    tot = sum(send)
                    ours_fn = lambda: cc.alltoallv(o, recv, i, send, stream=stream)  # noqa: E731
                elif coll == "reduce_scatter":
                    i, o = cc.empty(tot // 4, torch.float32), torch.empty(per // 4, device=dev)
                    i.fill_(1.0)
                    ours_fn = lambda: cc.reduce_scatter(o, i, stream=stream)  # noqa: E731
                    if nccl is not None:
                        nccl_fn = lambda: nccl.reduce_scatter(i.data_ptr(), o.data_ptr(), per // 4, F32, 1, stream.cuda_stream)  # noqa: E731
                else:
                    o = cc.empty(tot // 4, torch.float32)
                    i = None
                    bt = gcu.CudaBroadcastOneToAll(ctx, [o], root=0, streams=[stream])
                    ours_fn = bt.run
                    if nccl is not None:
                        nccl_fn = lambda: nccl.broadcast(o.data_ptr(), o.data_ptr(), tot // 4, F32, 0, stream.cuda_stream)  # noqa: E731
                torch.cuda.synchronize()
                p50, p99, _ = latency(ours_fn, iters, tot)
                factor = 1.0 if coll == "cuda_broadcast_one_to_all" else mv_factor
                row = {"bytes": tot, "p50_us": round(p50, 2), "p99_us": round(p99, 2),
                       "busbw_gbs": round(tot / (p50 * 1e-6) / 1e9 * factor, 3)}
                if nccl_fn is not None:
                    n50, _, _ = latency(nccl_fn, iters, tot)
                    row["nccl_p50_us"] = round(n50, 2)
                    row["nccl_busbw_gbs"] = round(tot / (n50 * 1e-6) / 1e9 * factor, 3)
                rows.append(row)
                del o, i
                torch.cuda.synchronize()
            configs[coll] = rows
        extra["peer_copy_gbs_measured_here"] = peer_copy_gbs

    # ---- latency sweep: per-iteration events, L2 flushed between iterations ----------------
    sweep = []
    if not args.no_sweep:
        iters = max(args.steps, 50)
        for n in SWEEP:
            ts, algo = make(n)
            with torch.cuda.stream(stream):
                fill_inputs(ts)
                algo.run()
            check_outputs(ts, f"sweep {n}")
            p50, p99, mn = latency(algo.run, iters, n * 4)
            ab = n * 4 / (p50 * 1e-6) / 1e9
            row = {"elements": n, "bytes": n * 4, "p50_us": round(p50, 2), "p99_us": round(p99, 2),
                   "min_us": round(mn, 2), "algbw_gbs": round(ab, 3),
                   "busbw_gbs": round(bus(ab), 3) if world > 1 else None,
                   "variant": algo.resolved_algo() if world > 1 else "local_fused"}
            if nccl is not None:
                ptr = ts[0].data_ptr()
                n50, n99, _ = latency(lambda: nccl.allreduce(ptr, ptr, n, F32, 1, stream.cuda_stream), iters, n * 4)
                row["nccl_p50_us"], row["nccl_p99_us"] = round(n50, 2), round(n99, 2)
            sweep.append(row)
            del ts, algo
    # ---- small messages inside a CUDA graph: 32 allreduces per graph, per-op time of a replay --------
    # (the per-iteration events above pay a launch + two event records per call; a training loop that
    # captures its step pays neither)
    graph_rows = []
    if not args.no_sweep and world > 1:
        OPS = 32
        for n in (1, 256, 4096):
            small = torch.ones(n, device=dev)
            row = {"elements": n, "bytes": n * 4, "ops_per_graph": OPS}
            for name in ("ours", "nccl"):
                if name == "nccl" and nccl is None:
                    continue
                try:
                    sync_all()
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=stream):
                        for _ in range(OPS):
                            if name == "ours":
                                cc.allreduce(small, stream=stream)
                            else:
                                nccl.allreduce(small.data_ptr(), small.data_ptr(), n, F32, 1, stream.cuda_stream)
                    p50, p99, mn = latency(g.replay, 30, n * 4)
                    key = "" if name == "ours" else "nccl_"
                    row[key + "p50_us_per_op"], row[key + "p99_us_per_op"] = round(p50 / OPS, 2), round(p99 / OPS, 2)
                    del g
                except Exception as e:  # noqa: BLE001
                    row[name + "_error"] = f"{type(e).__name__}: {str(e)[:120]}"
            graph_rows.append(row)
            del small
        extra["graph_small_allreduce"] = graph_rows
    sync_all()
    cc.check_health()
    del nccl
    if rank == 0:
        per_gpu = busbw if world > 1 else algbw
        value = per_gpu * world
        link = extra.get("peer_copy_gbs_measured_here")
        # Bytes that must cross NVLink per GPU and direction for this variant, against the link rate.
        wire_factor = {"nvls": (1 + 1 / world), "two_shot": 2 * (world - 1) / world}.get(resolved, None) if world > 1 else None
        if world > 1 and resolved == "hybrid":  # per-mille `tile` of the vector goes peer to peer, the rest through the switch
            pm = (plan.get("tile") or 175) / 1000.0
            wire_factor = (1 - pm) * (1 + 1 / world) + pm * 2 * (world - 1) / world
        roofline = {"nvlink_gbs_per_dir_nominal": 900,
                    "nvlink_gbs_per_dir_measured_guide": 770,
                    "nvlink_gbs_per_dir_measured_here": link,
                    "how": "measured_here = 256 MB one-directional put (our peerCopyKernel) to the next rank, device timed; "
                           "guide = /opt/skills/guides/B200_PROFILING.md (driver-measured peer copy)"}
        if wire_factor:
            wire = size_bytes * wire_factor / (ms_per_step * 1e-3) / 1e9
            roofline.update({"variant": resolved, "wire_bytes_per_gpu_per_dir": int(size_bytes * wire_factor),
                             "wire_gbs_per_dir": round(wire, 1), "frac_of_nominal": round(wire / 900, 3),
                             "frac_of_measured_guide": round(wire / 770, 3),
                             "frac_of_measured_here": round(wire / link, 3) if link else None})
        else:
            roofline.update({"variant": resolved, "hbm_gbs_measured": 6588.7,
                             "hbm_bytes_per_step": size_bytes * inputs * 2,
                             "frac_of_measured_hbm": round(size_bytes * inputs * 2 / (ms_per_step * 1e-3) / 1e9 / 6588.7, 3)})
        out = {
            "metric": METRIC,
            "value": round(value, 3), "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_per_step, 5), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": round(per_gpu / PUBLISHED_BUSBW_GBS, 2),
            "vs_baseline_basis": "per-GPU bus bandwidth / 2.8 GB/s (BASELINE.md: derived busbw of the published "
                                 "20 MB allreduce_ring_chunked row, 4 machines over 40 GbE)",
            "per_gpu_gbs": round(per_gpu, 3), "dtype": "fp32", "data": "synthetic",
            "impl": "gloo_b200",
            "config": {"model": "cuda_allreduce_ring_chunked", "elements": E, "bytes_per_gpu": size_bytes,
                       "inputs_per_rank": inputs, "global_batch": world * inputs, "seq_len": E,
                       "parallelism": f"allreduce x{world}", "cpu_affinity_cpus": len(cpus), "kernel_variant": resolved,
                       "launch_shape": plan, "tuning_table": cu.tuning_source(),
                       "buffers": "library symmetric allocator (peer-mapped; NVLS multicast-bound when >2 GPUs)",
                       "l2": "inputs larger than L2 (400 MB > 126 MB) for the headline; 256 MB flush between sweep iterations",
                       "timing": "CUDA events on the launching stream, max over ranks",
                       "verification": "whole buffer on every rank, device-side closed form, before and after the timed loop"},
            "algbw_gbs": round(algbw, 3), "busbw_gbs": round(busbw, 3) if busbw else None,
            "roofline": roofline,
            "clocks": clocks,
            "e2e": {"value": round(e2e_val * world, 3), "per_gpu_gbs": round(e2e_val, 3), "unit": "GB/s",
                    "ms_per_step": round(e2e_ms, 4),
                    "h2d_bytes_per_step": size_bytes * inputs, "d2h_bytes_per_step": size_bytes,
                    "api": "gloo_b200.ops.cuda.CudaHostAllreduce (chunked H2D | allreduce | D2H pipeline)",
                    "pieces": int(e2e_launches), "gpu_launches_per_step": int(e2e_launches)},
            "gpu_launches": int(launches),
            "verified": verified,
            **extra,
            "configs": configs,
            "sweep": sweep,
        }
        print(json.dumps(out), flush=True)
    ctx.close_connections()
    shutil.rmtree(rendezvous_dir("ours"), ignore_errors=True)


# ------------------------------------------------------------------------------------------
# reference arm: unmodified pytorch/gloo benchmark_cuda
# ------------------------------------------------------------------------------------------

ROW = re.compile(r"^\s*(\d+)\s+(\d+)\s+(\d+)\s+(\d+)\s+(\d+)\s+(\d+)\s+([0-9.]+)\s+(\d+)\s*$")


def run_reference(args):
    rank, world = env_int("RANK", 0), env_int("WORLD_SIZE", 1)
    local = env_int("LOCAL_RANK", 0)
    bindir = os.path.join(ROOT, "baseline", "_ref", "bin")
    binary = os.path.join(bindir, "benchmark_cuda")
    if not os.path.exists(binary):
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref/bin/benchmark_cuda missing "
                              "(pip cannot install the CMake-only reference; build it with baseline/build_reference.sh)"}))
        return
    # The reference cannot place two inputs on one GPU (its local reduce goes through NCCL,
    # which needs unique devices: nccl.cu:111-116), so its 1-GPU run uses one buffer and
    # does D2H + H2D of it; our 1-GPU run reduces and re-broadcasts two buffers (more work).
    inputs = 1
    base = rendezvous_dir("ref")
    env = dict(os.environ)
    env["CUDA_VISIBLE_DEVICES"] = str(local)
    seq = [0]

    def one(elements, iters, warmup, name="cuda_allreduce_ring_chunked", extra_flags=(), exe=binary):
        seq[0] += 1
        d = f"{base}_{seq[0]}"
        os.makedirs(d, exist_ok=True)
        cmd = [exe, "--size", str(world), "--rank", str(rank), "--shared-path", d, "--transport", "tcp",
               "--tcp-device", "lo", "--elements", str(elements), "--iteration-count", str(iters),
               "--warmup-iters", str(warmup), "--inputs", str(inputs), "--no-verify", "--nanos", *extra_flags, name]
        p = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=1500)
        row = None
        for ln in p.stdout.splitlines():
            m = ROW.match(ln)
            if m:
                row = [float(x) for x in m.groups()]
        if p.returncode != 0 or (rank == 0 and row is None):
            raise RuntimeError(f"reference {name} failed (rc={p.returncode}): {p.stderr[-400:]} {p.stdout[-400:]}")
        return row

    def mean_ms(row):
        # Mean latency from the reference's own bandwidth column (GiB/s over the sum of
        # latencies, runner.cc:499-508); fall back to p50 when the column underflows.
        size_bytes, _, mn, p50, p99, mx, bw_gib, iters = row
        ns = size_bytes / (bw_gib * (1 << 30)) * 1e9 if bw_gib > 0 else p50
        return ns / 1e6

    ar = 2 * (world - 1) / world if world > 1 else 1.0
    configs = {}
    e2e = None
    try:
        head = one(args.elements, args.steps, args.warmup)
        sweep = []
        if not args.no_sweep:
            for n in (1_000, 100_000, 1_000_000, 10_000_000):
                r = one(n, max(args.steps, 20), max(args.warmup, 3))
                if rank == 0:
                    p50 = r[3] / 1e3
                    ab = n * 4 / (p50 * 1e-6) / 1e9
                    sweep.append({"elements": n, "bytes": n * 4, "p50_us": round(p50, 2), "p99_us": round(r[4] / 1e3, 2),
                                  "min_us": round(r[2] / 1e3, 2), "algbw_gbs": round(ab, 4),
                                  "busbw_gbs": round(ab * 2 * (world - 1) / world, 4) if world > 1 else None})
        if not args.quick and world > 1:
            # BASELINE config 3 (fp16 halving-doubling / bcube) and config 5 (broadcast), stock benchmark_cuda.
            for key, name in (("cuda_allreduce_halving_doubling_fp16", "cuda_allreduce_halving_doubling"),
                              ("cuda_allreduce_bcube_fp16", "cuda_allreduce_bcube")):
                rows = []
                for n in (100_000, 10_000_000):
                    r = one(n, 5, 2, name=name, extra_flags=("--halfprecision",))
                    if rank == 0:
                        ms = mean_ms(r)
                        rows.append({"elements": n, "bytes": n * 2, "ms": round(ms, 4),
                                     "busbw_gbs": round(n * 2 / (ms * 1e-3) / 1e9 * ar, 4)})
                configs[key] = rows
            rows = []
            for n in (256, 1 << 20, 64 << 20):  # float32 elements: 1 KB, 4 MB, 256 MB
                r = one(n, 5, 2, name="cuda_broadcast_one_to_all")
                if rank == 0:
                    ms = mean_ms(r)
                    rows.append({"bytes": n * 4, "p50_us": round(r[3] / 1e3, 2), "busbw_gbs": round(n * 4 / (ms * 1e-3) / 1e9, 4)})
            configs["cuda_broadcast_one_to_all"] = rows
            # BASELINE config 4 + reduce_scatter: host buffers only in the reference (no CUDA variant exists).
            host = os.path.join(bindir, "benchmark")
            if os.path.exists(host):
                for key, name in (("allgather", "allgather"), ("alltoall", "alltoall"), ("reduce_scatter", "reduce_scatter")):
                    rows = []
                    for n in (256, 16384, 1 << 20):
                        try:
                            r = one(n, 10, 2, name=name, exe=host)
                        except Exception:  # noqa: BLE001
                            break
                        if rank == 0:
                            rows.append({"elements_per_rank": n, "p50_us": round(r[3] / 1e3, 2), "note": "host buffers"})
                    configs[key] = rows
        # End to end: pinned host -> GPU -> stock CudaAllreduceRingChunked::run() -> pinned host.
        exe = os.path.join(bindir, "ref_e2e")
        if os.path.exists(exe):
            d = f"{base}_e2e"
            os.makedirs(d, exist_ok=True)
            p = subprocess.run([exe, "--size", str(world), "--rank", str(rank), "--shared-path", d, "--elements",
                                str(args.elements), "--steps", str(max(3, min(args.steps, 10))), "--warmup", "2"],
                               env=env, capture_output=True, text=True, timeout=1500)
            m = re.search(r"ms_per_step=([0-9.]+)", p.stdout)
            if p.returncode == 0 and m:
                # every rank writes its number; rank 0 takes the max (same convention as our arm)
                with open(os.path.join(d, f"done_{rank}"), "w") as f:
                    f.write(m.group(1))
                if rank == 0:
                    vals, deadline = [], time.time() + 120
                    for r in range(world):
                        fp = os.path.join(d, f"done_{r}")
                        while not os.path.exists(fp) or os.path.getsize(fp) == 0:
                            if time.time() > deadline:
                                break
                            time.sleep(0.05)
                        if os.path.exists(fp):
                            vals.append(float(open(fp).read() or 0))
                    ms = max(vals) if vals else float(m.group(1))
                    algbw = args.elements * 4 / (ms * 1e-3) / 1e9
                    pg = algbw * ar if world > 1 else algbw
                    e2e = {"value": round(pg * world, 4), "per_gpu_gbs": round(pg, 4), "unit": "GB/s", "ms_per_step": round(ms, 4),
                           "h2d_bytes_per_step": args.elements * 4, "d2h_bytes_per_step": args.elements * 4,
                           "api": "baseline/ref_e2e.cc: cudaMemcpyAsync H2D -> gloo::CudaAllreduceRingChunked<float>::run() "
                                  "(stock CudaHostWorkspace) -> cudaMemcpyAsync D2H, host wall clock, max over ranks"}
            elif rank == 0:
                e2e = {"unavailable": f"ref_e2e rc={p.returncode}: {(p.stderr or p.stdout)[-200:]}"}
    except Exception as e:  # noqa: BLE001
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": f"reference run failed: {str(e)[:300]}"}))
        return
    if rank == 0:
        size_bytes, _, mn, p50, p99, mx, bw_gib, iters = head
        ms = mean_ms(head)
        algbw = size_bytes / (ms * 1e-3) / 1e9
        per_gpu = algbw * 2 * (world - 1) / world if world > 1 else algbw
        value = per_gpu * world
        out = {
            "metric": METRIC,
            "value": round(value, 4), "unit": "GB/s", "n_gpus": world, "steps": int(iters), "warmup": args.warmup,
            "ms_per_step": round(ms, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": round(per_gpu / PUBLISHED_BUSBW_GBS, 3), "per_gpu_gbs": round(per_gpu, 4),
            "dtype": "fp32", "data": "synthetic",
            "impl": "reference",
            "config": {"model": "cuda_allreduce_ring_chunked", "elements": args.elements, "bytes_per_gpu": int(size_bytes),
                       "inputs_per_rank": inputs, "global_batch": world * inputs, "seq_len": args.elements,
                       "parallelism": f"allreduce x{world}",
                       "timing": "reference's own harness: host wall clock on rank 0 (runner.cc:641-645), "
                                 "mean from its bandwidth column",
                       "path": "pytorch/gloo benchmark_cuda (CudaHostWorkspace: GPU->pinned host->TCP loopback->CPU reduce)"},
            "p50_us": round(p50 / 1e3, 2), "p99_us": round(p99 / 1e3, 2), "configs": configs, "sweep": sweep,
        }
        if e2e is not None:
            out["e2e"] = e2e
        print(json.dumps(out), flush=True)
    if rank == 0:  # only rank 0: the others may finish while it still reads the e2e files
        for d in glob.glob(base + "_*"):
            shutil.rmtree(d, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--elements", type=int, default=HEADLINE_ELEMENTS)
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline + e2e + latency sweep only (skip BASELINE configs 3-5)")
    ap.add_argument("--no-verify-matrix", action="store_true", help="skip the multi-GPU correctness matrix before timing")
    ap.add_argument("--e2e-chunks", type=int, default=16, help="pieces of the host<->device pipeline in the e2e run")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the buffers of the last timed headline step to DIR/*.npy (float32, seeded sample "
                         f"when they exceed {DUMP_BYTES >> 20} MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
