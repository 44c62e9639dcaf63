"""CUDA-buffer collectives over NVLink peer memory.

``CudaContext`` wraps the native PeerContext (topology exchange + symmetric pool)
and offers the collective suite for torch CUDA tensors. A tensor is either

* *registered* (``ctx.register(t)`` or allocated with ``ctx.empty(...)``): kernels
  read/write the peers' copies directly (zero-copy, NVLS-capable when symmetric);
* anything else: staged through the pool inside the same call.

Every method is asynchronous on the current torch stream unless ``stream`` is given,
and must be called in the same order on every rank.
"""
from __future__ import annotations

import weakref
from typing import Any, Dict, List, Optional, Sequence, Tuple

from .. import _C
from ..types import DataType, ReduceOp, describe, element_size

_cu = _C.cuda

ALGOS = {"auto": 0, "one_shot": 1, "two_shot": 2, "nvls": 3, "ll": 4, "pipelined": 5, "hybrid": 6, "ring": 10, "ring_chunked": 11,
         "halving_doubling": 12, "bcube": 13, "halving_doubling_pipelined": 14}


def _torch_dtype_to_glb(dtype) -> DataType:
    import torch

    return {torch.float32: DataType.FLOAT32, torch.float16: DataType.FLOAT16, torch.bfloat16: DataType.BFLOAT16,
            torch.float64: DataType.FLOAT64}[dtype]


def _stream(stream) -> int:
    if stream is None:
        import torch

        return torch.cuda.current_stream().cuda_stream
    if isinstance(stream, int):
        return stream
    return stream.cuda_stream


def _algo(a) -> int:
    return ALGOS[a] if isinstance(a, str) else int(a)


# (input, output) dtypes that reduce_scatter / allgather(v) convert inside the kernel
CAST_PAIRS = frozenset({(DataType.FLOAT32, DataType.FLOAT16), (DataType.FLOAT32, DataType.BFLOAT16),
                        (DataType.FLOAT16, DataType.FLOAT32), (DataType.BFLOAT16, DataType.FLOAT32)})


def _cast_types(what: str, in_dtype, out_dtype) -> Tuple[DataType, DataType]:
    """DataTypes of a converting call from torch dtypes ``in_dtype`` -> ``out_dtype`` (which
    differ); TypeError for any pair outside ``CAST_PAIRS``. Same-dtype calls never come here: they
    move raw bytes of any dtype, including those without a DataType (float8, complex, uint16...)."""
    try:
        pair = (_torch_dtype_to_glb(in_dtype), _torch_dtype_to_glb(out_dtype))
    except KeyError:
        pair = None
    if pair not in CAST_PAIRS:
        raise TypeError(f"{what}: cannot convert {in_dtype} to {out_dtype}; the supported conversions are "
                        "FLOAT32 -> FLOAT16 / BFLOAT16 and FLOAT16 / BFLOAT16 -> FLOAT32")
    return pair


def _check_counts(what: str, counts: Sequence[int], size: int) -> List[int]:
    counts = [int(c) for c in counts]
    if len(counts) != size or any(c < 0 for c in counts):
        raise ValueError(f"{what}: need {size} non-negative element counts, got {counts}")
    return counts


def _check_len(what: str, name: str, have: int, need: int) -> None:
    if have < need:
        raise ValueError(f"{what}: {name} holds {have} elements, the counts need {need}")


def new_stream(device: Optional[int] = None, high_priority: bool = False):
    """A dedicated CUDA stream as a torch ExternalStream (never shared through torch's pool)."""
    import torch

    device = torch.cuda.current_device() if device is None else device
    raw = _cu.create_stream(int(device), high_priority)
    return torch.cuda.ExternalStream(raw, device=device)


class _SymmetricStorage:
    """Exposes a PeerBuffer through __cuda_array_interface__ so torch can wrap it."""

    def __init__(self, buf, nbytes: int):
        self.buf = buf
        self.__cuda_array_interface__ = {
            "shape": (nbytes,), "typestr": "|u1", "data": (buf.ptr, False), "version": 3, "strides": None,
        }


class CudaContext:
    def __init__(self, ctx, device: Optional[int] = None, stage_bytes: int = 0, use_vmm: bool = True,
                 use_nvls: bool = True):
        import torch

        if device is None:
            device = torch.cuda.current_device()
        self.ctx = ctx
        self.device = int(device)
        with torch.cuda.device(self.device):
            # One PeerContext per (context, device), shared with the old-style CUDA classes
            # (it is an attachment of the context): symmetric tensors allocated here are
            # recognised by CudaAllreduce* / CudaBroadcastOneToAll and get the NVLS path.
            self.pc = _cu.peer_context_for(ctx, self.device, stage_bytes, use_vmm, use_nvls)
        self.rank, self.size = self.pc.rank, self.pc.size
        # base ptr -> (PeerBuffer | weakref to the symmetric storage, nbytes)
        self._reg: Dict[int, Tuple[Any, int]] = {}

    # ---- memory -------------------------------------------------------------------------
    def register(self, tensor):
        """Collective: make ``tensor``'s memory addressable by every rank."""
        ptr, n, dt, cuda = describe(tensor)
        assert cuda, "register() needs a CUDA tensor"
        nbytes = n * element_size(dt)
        buf = self.pc.register_buffer(ptr, nbytes)
        self._reg[ptr] = (buf, nbytes)
        return buf

    def empty(self, shape, dtype):
        """Collective: allocate a symmetric tensor (peer-mapped, NVLS-bound when available)."""
        import math

        import torch

        shape = (shape,) if isinstance(shape, int) else tuple(shape)
        n = math.prod(shape)
        es = torch.empty((), dtype=dtype).element_size()
        nbytes = max(16, n * es)
        buf = self.pc.alloc_symmetric(nbytes)
        store = _SymmetricStorage(buf, nbytes)
        flat = torch.as_tensor(store, device=f"cuda:{self.device}")
        t = flat[: n * es].view(dtype).view(shape)
        # The tensor keeps `store` (and through it the PeerBuffer) alive; when the last view
        # dies the symmetric memory and its multicast binding are released.
        self._reg[buf.ptr] = (weakref.ref(store), nbytes)
        return t

    def lookup(self, tensor) -> Tuple[Optional[Any], int]:
        """(PeerBuffer, byte offset) if ``tensor`` lies inside a registered region."""
        ptr = tensor.data_ptr()
        nbytes = tensor.numel() * tensor.element_size()
        dead = []
        found = (None, 0)
        for base, (ref, size) in self._reg.items():
            buf = ref
            if isinstance(ref, weakref.ref):
                store = ref()
                if store is None:
                    dead.append(base)
                    continue
                buf = store.buf
            if base <= ptr and ptr + nbytes <= base + size:
                found = (buf, ptr - base)
                break
        for b in dead:
            del self._reg[b]
        return found

    # ---- info ---------------------------------------------------------------------------
    def describe(self) -> str:
        return self.pc.describe()

    def topology(self):
        return self.pc.topology()

    def nvls_available(self) -> bool:
        return self.pc.nvls_available()

    # ---- collectives ----------------------------------------------------------------------
    def barrier(self, stream=None):
        _cu.barrier(self.pc, _stream(stream))

    def allreduce(self, tensor, op: ReduceOp = ReduceOp.SUM, algo="auto", out=None, stream=None, scale: float = 1.0,
                  average: bool = False, extra: Sequence = (), blocks: int = 0, unroll: int = 0, tile: int = 0):
        """In place on ``tensor`` (or tensor -> out), ONE kernel launch.

        ``scale`` / ``average`` (= 1/size) are applied to the fp32 accumulator inside the
        collective kernel, before the single rounding to the output dtype. ``out`` may have a
        different dtype (float32 <-> float16 / bfloat16): registered tensors of any size, plain
        tensors up to the LL limit. ``extra``: more local tensors of the same shape that are
        folded into the reduction and overwritten with the result (multi-pointer semantics).
        ``blocks`` / ``unroll`` / ``tile`` pin the launch shape (tuner)."""
        ptr, n, dt, _ = describe(tensor)
        s = _stream(stream)
        if average:
            scale = scale / self.size
        ex = [t.data_ptr() for t in extra]
        if out is None or out.data_ptr() == ptr:
            buf, off = self.lookup(tensor)
            if buf is not None:
                _cu.allreduce_registered(self.pc, buf, off, n, int(dt), int(op), _algo(algo), s, scale, ex, blocks,
                                         unroll, tile)
                return tensor
            _cu.allreduce(self.pc, ptr, ptr, n, int(dt), int(op), _algo(algo), s, scale, -1, ex, blocks, tile, unroll)
            return tensor
        _, _, odt, _ = describe(out)
        if odt != dt:
            ibuf, ioff = self.lookup(tensor)
            obuf, ooff = self.lookup(out)
            if ibuf is not None and obuf is not None and not ex:
                _cu.allreduce_cast(self.pc, ibuf, ioff, obuf, ooff, n, int(dt), int(odt), int(op), s, scale, blocks)
                return out
            _cu.allreduce(self.pc, ptr, out.data_ptr(), n, int(dt), int(op), _algo(algo), s, scale, int(odt), ex, blocks,
                          tile, unroll)
            return out
        _cu.allreduce(self.pc, ptr, out.data_ptr(), n, int(dt), int(op), _algo(algo), s, scale, -1, ex, blocks, tile, unroll)
        return out

    def plan(self, tensor, op: ReduceOp = ReduceOp.SUM) -> dict:
        """What ``algo="auto"`` resolves to for this tensor (variant + launch shape)."""
        _, n, dt, _ = describe(tensor)
        buf, off = self.lookup(tensor)
        kind = 2 if buf is None else (0 if (buf.has_multicast and off % 16 == 0) else 1)
        return _cu.plan_allreduce(self.pc, n * element_size(dt), int(dt), int(op), kind)

    # ---- health ---------------------------------------------------------------------------
    def set_timeout(self, ms: int):
        """Device-side waits give up after ``ms`` milliseconds (then the context is poisoned)."""
        self.pc.set_timeout(int(ms))

    def check_health(self):
        self.pc.check_health()

    def synchronize(self, stream=None):
        """Wait for the stream and raise ``IoException`` if a peer went missing meanwhile."""
        self.pc.synchronize(_stream(stream))

    # ---- point to point ---------------------------------------------------------------------
    def send(self, tensor, dst: int, stream=None):
        """Stream ``tensor`` to rank ``dst`` over NVLink (matched with its recv in posting order)."""
        _cu.send(self.pc, tensor.data_ptr(), tensor.numel() * tensor.element_size(), dst, _stream(stream))

    def recv(self, tensor, src: int, stream=None):
        _cu.recv(self.pc, tensor.data_ptr(), tensor.numel() * tensor.element_size(), src, _stream(stream))
        return tensor

    def sendrecv(self, send_tensor, dst: int, recv_tensor, src: int, stream=None):
        """Both directions in one kernel: the call for ring / pipeline exchanges."""
        _cu.sendrecv(self.pc, send_tensor.data_ptr(), send_tensor.numel() * send_tensor.element_size(), dst,
                     recv_tensor.data_ptr(), recv_tensor.numel() * recv_tensor.element_size(), src, _stream(stream))
        return recv_tensor

    def exchange(self, send_tensor, dst: int, recv_tensor, src: int, stream=None):
        """Zero-copy sendrecv: ``recv_tensor`` is a registered / symmetric tensor that EVERY rank passes at the
        same offset; my payload is written straight into ``dst``'s copy of it, ``src`` writes into mine.

        One kernel and one pass over the data (sendrecv() stages through a mailbox ring). Falls back to
        sendrecv() when ``recv_tensor`` is not registered."""
        buf, off = self.lookup(recv_tensor)
        if buf is None:
            return self.sendrecv(send_tensor, dst, recv_tensor, src, stream)
        _cu.exchange(self.pc, send_tensor.data_ptr(), send_tensor.numel() * send_tensor.element_size(), dst, buf, off,
                     recv_tensor.numel() * recv_tensor.element_size(), src, _stream(stream))
        return recv_tensor

    def put(self, local, remote, peer: int, remote_offset: int = 0, stream=None):
        """One-sided: copy ``local`` into rank ``peer``'s copy of the registered tensor ``remote``."""
        buf, off = self.lookup(remote)
        assert buf is not None, "put() needs a registered / symmetric remote tensor"
        _cu.put(self.pc, local.data_ptr(), buf, off + remote_offset * remote.element_size(),
                local.numel() * local.element_size(), peer, _stream(stream))

    def get(self, local, remote, peer: int, remote_offset: int = 0, stream=None):
        """One-sided: read rank ``peer``'s copy of the registered tensor ``remote`` into ``local``."""
        buf, off = self.lookup(remote)
        assert buf is not None, "get() needs a registered / symmetric remote tensor"
        _cu.get(self.pc, local.data_ptr(), buf, off + remote_offset * remote.element_size(),
                local.numel() * local.element_size(), peer, _stream(stream))
        return local

    def broadcast(self, tensor, root: int = 0, stream=None):
        ptr, n, dt, _ = describe(tensor)
        nbytes = n * element_size(dt)
        buf, off = self.lookup(tensor)
        if buf is not None:
            _cu.broadcast_reg(self.pc, buf, off, nbytes, root, _stream(stream))
        else:
            _cu.broadcast(self.pc, ptr, nbytes, root, _stream(stream))
        return tensor

    def allgather(self, output, input, stream=None):
        """Every rank's ``input`` (same length on every rank), in rank order, in every ``output``.
        ``output`` may have another dtype than ``input``: see ``allgatherv``."""
        return self.allgatherv(output, input, [input.numel()] * self.size, stream)

    def allgatherv(self, output, input, counts: Sequence[int], stream=None):
        """Rank r's ``input`` (``counts[r]`` elements) lands at element offset ``sum(counts[:r])`` of
        every rank's ``output``.

        With ``output.dtype != input.dtype`` (float32 -> float16 / bfloat16, or float16 / bfloat16 ->
        float32) each rank's block is converted once inside the kernel: narrowing rounds to nearest
        even (values beyond the float16 range become Inf), widening is exact. Only the output dtype
        crosses NVLink. Raises ``ValueError`` when ``output`` or ``input`` is shorter than the counts
        say and ``TypeError`` for any other dtype pair, before anything is launched."""
        counts = _check_counts("allgatherv", counts, self.size)
        _check_len("allgatherv", "output", output.numel(), sum(counts))
        _check_len("allgatherv", "input", input.numel() if input is not None else 0, counts[self.rank])
        buf, off = self.lookup(output)
        iptr = input.data_ptr() if input is not None else 0
        if input is not None and input.dtype != output.dtype:
            idt, odt = _cast_types("allgatherv", input.dtype, output.dtype)
            if buf is not None:
                _cu.allgatherv_cast_reg(self.pc, iptr, int(idt), buf, off, counts, int(odt), _stream(stream))
            else:
                _cu.allgatherv_cast(self.pc, iptr, int(idt), output.data_ptr(), counts, int(odt), _stream(stream))
            return output
        es = output.element_size()
        sizes = [c * es for c in counts]
        if buf is not None:
            _cu.allgatherv_reg(self.pc, iptr, buf, off, sizes, _stream(stream))
        else:
            _cu.allgatherv(self.pc, iptr, output.data_ptr(), sizes, _stream(stream))
        return output

    def gather(self, output, input, root: int = 0, stream=None):
        return self.gatherv(output, input, [input.numel()] * self.size, root, stream)

    def gatherv(self, output, input, counts: Sequence[int], root: int = 0, stream=None):
        es = input.element_size()
        sizes = [int(c) * es for c in counts]
        optr = output.data_ptr() if output is not None else 0
        buf, off = (self.lookup(output) if output is not None else (None, 0))
        if buf is not None:
            _cu.gatherv_reg(self.pc, input.data_ptr(), buf, off, sizes, root, _stream(stream))
        else:
            _cu.gatherv(self.pc, input.data_ptr(), optr, sizes, root, _stream(stream))
        return output

    def alltoall(self, output, input, stream=None):
        """Fixed-size exchange: chunk j of ``input`` goes to rank j (one size for all ranks)."""
        per = input.numel() // self.size * input.element_size()
        buf, off = self.lookup(output)
        if buf is not None:
            _cu.alltoall_reg(self.pc, input.data_ptr(), buf, off, per, _stream(stream))
        else:
            _cu.alltoall(self.pc, input.data_ptr(), output.data_ptr(), per, _stream(stream))
        return output

    def alltoallv(self, output, out_counts: Sequence[int], input, in_counts: Sequence[int], stream=None):
        es = input.element_size()
        send = [int(c) * es for c in in_counts]
        recv = [int(c) * es for c in out_counts]
        buf, off = self.lookup(output)
        if buf is not None:
            _cu.alltoallv_reg(self.pc, input.data_ptr(), send, buf, off, recv, _stream(stream))
        else:
            _cu.alltoallv(self.pc, input.data_ptr(), send, output.data_ptr(), recv, _stream(stream))
        return output

    def scatter(self, output, input=None, root: int = 0, stream=None):
        nbytes = output.numel() * output.element_size()
        iptr = input.data_ptr() if input is not None else 0
        buf, off = self.lookup(output)
        if buf is not None:
            _cu.scatter_reg(self.pc, iptr, buf, off, nbytes, root, _stream(stream))
        else:
            _cu.scatter(self.pc, iptr, output.data_ptr(), nbytes, root, _stream(stream))
        return output

    def reduce_scatter(self, output, input, counts: Optional[Sequence[int]] = None, op: ReduceOp = ReduceOp.SUM,
                       stream=None, scale: float = 1.0):
        """Rank r gets elements ``[sum(counts[:r]), +counts[r])`` of the reduction of every rank's
        ``input`` in ``output`` (default counts: ``input`` split as evenly as possible).

        With ``output.dtype != input.dtype`` (float32 -> float16 / bfloat16, or float16 / bfloat16 ->
        float32) the kernel accumulates in float32, multiplies the accumulator by ``scale`` and rounds
        once to the output dtype; the input dtype is what crosses NVLink. Raises ``ValueError`` when
        ``output`` or ``input`` is shorter than the counts say and ``TypeError`` for any other dtype
        pair, before anything is launched."""
        cast = _cast_types("reduce_scatter", input.dtype, output.dtype) if output.dtype != input.dtype else None
        ptr, n, dt, _ = describe(input)
        if counts is None:
            base, rem = divmod(n, self.size)
            counts = [base + (1 if r < rem else 0) for r in range(self.size)]
        counts = _check_counts("reduce_scatter", counts, self.size)
        _check_len("reduce_scatter", "input", n, sum(counts))
        _check_len("reduce_scatter", "output", output.numel(), counts[self.rank])
        buf, off = self.lookup(input)
        if cast is not None:
            odt = cast[1]
            if buf is not None:
                _cu.reduce_scatter_cast_reg(self.pc, buf, off, output.data_ptr(), counts, int(dt), int(odt), int(op),
                                            _stream(stream), scale)
            else:
                _cu.reduce_scatter_cast(self.pc, ptr, output.data_ptr(), counts, int(dt), int(odt), int(op),
                                        _stream(stream), scale)
            return output
        if buf is not None:
            _cu.reduce_scatter_reg(self.pc, buf, off, output.data_ptr(), counts, int(dt), int(op), _stream(stream), scale)
        else:
            _cu.reduce_scatter(self.pc, ptr, output.data_ptr(), counts, int(dt), int(op), _stream(stream), scale)
        return output

    def reduce(self, output, input, root: int = 0, op: ReduceOp = ReduceOp.SUM, stream=None):
        ptr, n, dt, _ = describe(input)
        ibuf, ioff = self.lookup(input)
        obuf, ooff = (self.lookup(output) if output is not None else (None, 0))
        if ibuf is not None and obuf is not None:
            _cu.reduce_reg(self.pc, ibuf, ioff, obuf, ooff, n, int(dt), int(op), root, _stream(stream))
        else:
            optr = output.data_ptr() if output is not None else 0
            _cu.reduce(self.pc, ptr, optr, n, int(dt), int(op), root, _stream(stream))
        return output


# ---- old-style class wrappers -----------------------------------------------------------------

def _make_allreduce_class(name: str, algo: str):
    class _Cls:
        __doc__ = f"{name}(ctx, tensors, streams=None, op=SUM, host_workspace=False) — run() is one fused launch."

        def __init__(self, ctx, tensors, streams=None, op: ReduceOp = ReduceOp.SUM, host_workspace: bool = False,
                     literal: bool = False, variant: str = "auto"):
            # literal=True runs the named schedule step by step; otherwise the kernel variant is
            # picked per message size ("auto") or pinned ("one_shot" / "two_shot" / "nvls").
            tensors = list(tensors) if isinstance(tensors, (list, tuple)) else [tensors]
            self.tensors = tensors
            _, n, dt, _ = describe(tensors[0])
            st = [_stream(s) for s in streams] if streams else []
            assert variant in ("auto", "one_shot", "two_shot", "nvls", "ll", "pipelined", "hybrid")
            self._impl = _cu.CudaAllreduce(ctx, [t.data_ptr() for t in tensors], n, int(dt), int(op), st,
                                           ALGOS[algo] if literal else ALGOS[variant], host_workspace)

        def run(self):
            self._impl.run()

        def set_scale(self, scale: float):
            """Fused epilogue: the result is multiplied by ``scale`` inside the collective kernel."""
            self._impl.set_scale(float(scale))

        def set_launch_shape(self, blocks: int = 0, unroll: int = 0, tile: int = 0):
            self._impl.set_launch_shape(blocks, unroll, tile)

        def launches_per_run(self) -> int:
            return self._impl.launches_per_run()

        def resolved_algo(self) -> str:
            return self._impl.resolved_algo()

        def uses_peer_memory(self) -> bool:
            return self._impl.uses_peer_memory()

    _Cls.__name__ = name
    return _Cls


CudaAllreduceRing = _make_allreduce_class("CudaAllreduceRing", "ring")
CudaAllreduceRingChunked = _make_allreduce_class("CudaAllreduceRingChunked", "ring_chunked")
CudaAllreduceHalvingDoubling = _make_allreduce_class("CudaAllreduceHalvingDoubling", "halving_doubling")
CudaAllreduceHalvingDoublingPipelined = _make_allreduce_class("CudaAllreduceHalvingDoublingPipelined",
                                                              "halving_doubling_pipelined")
CudaAllreduceBcube = _make_allreduce_class("CudaAllreduceBcube", "bcube")


class CudaHostAllreduce:
    """Allreduce of pinned *host* buffers through the GPUs, as a three-stage pipeline.

    The reference reaches host-resident data with ``CudaHostWorkspace`` (device <-> pinned host
    staging around a CPU reduction, gloo/cuda_workspace.h:17-40). Here the reduction stays on
    NVLink and the PCIe legs are overlapped with it: the vector is cut into ``chunks`` pieces and
    piece c is copied host->device on one stream while piece c-1 is being reduced across the
    GPUs (one fused kernel per piece, same ``CudaAllreduceRingChunked`` class a user would
    call) and piece c-2 is copied device->host on a third stream. PCIe is full duplex, so a
    step costs about max(H2D, D2H) + one piece instead of H2D + allreduce + D2H.

    ``host_inputs``: one pinned tensor per local input (they are summed first when there are
    several, like the multi-pointer classes); ``host_output``: pinned tensor for the result.
    ``run()`` is asynchronous with respect to the host: the caller's current stream (or
    ``stream``) is made to wait for the last device->host copy, so ``stream.synchronize()``
    or any later work on that stream sees ``host_output`` complete. Collective: construct
    and run in the same order on every rank.
    """

    def __init__(self, ctx, cuda_ctx: "CudaContext", host_inputs, host_output, chunks: int = 16,
                 op: ReduceOp = ReduceOp.SUM, variant: str = "two_shot"):
        import torch

        host_inputs = list(host_inputs) if isinstance(host_inputs, (list, tuple)) else [host_inputs]
        n = host_output.numel()
        for h in host_inputs + [host_output]:
            assert h.is_pinned() and h.is_contiguous() and h.numel() == n and h.dtype == host_output.dtype, \
                "CudaHostAllreduce needs contiguous pinned host tensors of one shape and dtype"
        self.cc = cuda_ctx
        self.hin, self.hout = host_inputs, host_output
        dev = cuda_ctx.device
        with torch.cuda.device(dev):
            self.dev = [cuda_ctx.empty(n, host_output.dtype) for _ in host_inputs]
            self.h2d, self.comp, self.d2h = new_stream(dev), new_stream(dev, True), new_stream(dev)
            # piece boundaries on 4 KiB so every piece keeps the vector alignment of the kernels
            align = max(1, 4096 // host_output.element_size())
            per = -(-n // max(1, chunks))
            per = -(-per // align) * align
            self.bounds = [(lo, min(n, lo + per)) for lo in range(0, n, per)] if n else []
            self.algos = []
            for lo, hi in self.bounds:
                # Pieces are interior ranges of the symmetric buffers. The two-shot kernel is
                # pinned: it is the variant measured on such ranges, and the reduction hides
                # under the PCIe copies either way.
                self.algos.append(CudaAllreduceRingChunked(ctx, [d[lo:hi] for d in self.dev],
                                                           streams=[self.comp] * len(self.dev), op=op,
                                                           variant=variant))
            self.ev_in = [torch.cuda.Event() for _ in self.bounds]
            self.ev_red = [torch.cuda.Event() for _ in self.bounds]
            self.ev_start, self.ev_done = torch.cuda.Event(), torch.cuda.Event()
        self.launches_per_run = len(self.bounds)

    def run(self, stream=None):
        import torch

        caller = torch.cuda.current_stream(self.cc.device) if stream is None else stream
        self.ev_start.record(caller)
        self.h2d.wait_event(self.ev_start)
        self.d2h.wait_event(self.ev_start)
        for c, (lo, hi) in enumerate(self.bounds):
            with torch.cuda.stream(self.h2d):
                for d, h in zip(self.dev, self.hin):
                    d[lo:hi].copy_(h[lo:hi], non_blocking=True)
                self.ev_in[c].record(self.h2d)
            self.comp.wait_event(self.ev_in[c])
            self.algos[c].run()
            self.ev_red[c].record(self.comp)
            self.d2h.wait_event(self.ev_red[c])
            with torch.cuda.stream(self.d2h):
                self.hout[lo:hi].copy_(self.dev[0][lo:hi], non_blocking=True)
        self.ev_done.record(self.d2h)
        caller.wait_event(self.ev_done)
        return self.hout

    def resolved_algo(self) -> str:
        return self.algos[0].resolved_algo() if self.algos else "none"


class CudaBroadcastOneToAll:
    def __init__(self, ctx, tensors, root: int = 0, root_pointer: int = 0, streams=None, host_workspace: bool = False):
        tensors = list(tensors) if isinstance(tensors, (list, tuple)) else [tensors]
        self.tensors = tensors
        _, n, dt, _ = describe(tensors[0])
        st = [_stream(s) for s in streams] if streams else []
        self._impl = _cu.CudaBroadcast(ctx, [t.data_ptr() for t in tensors], n, int(dt), root, root_pointer, st,
                                       host_workspace)

    def run(self):
        self._impl.run()
