from __future__ import annotations

from typing import Iterable, List, Optional, Sequence

from .. import _C
from ..ops import host as H
from ..types import ReduceOp


def _is_cuda(t) -> bool:
    return bool(getattr(t, "is_cuda", False))


class _Base:
    def __init__(self, ctx, cuda_ctx=None):
        """ctx: host context (control plane, CPU tensors); cuda_ctx: ops.cuda.CudaContext."""
        self.ctx = ctx
        self.cc = cuda_ctx
        self.rank, self.size = ctx.rank, ctx.size

    def _allreduce(self, t, op=ReduceOp.SUM, average: bool = False):
        """Allreduce, optionally averaged. On CUDA the 1/P is the kernel's fused scale epilogue
        (one launch); on the host it is a second pass."""
        if _is_cuda(t):
            fused = average and t.is_floating_point()
            self.cc.allreduce(t, op=op, average=fused)
            if average and not fused:
                t.div_(self.size)
        else:
            H.allreduce(self.ctx, t, op=op)
            if average:
                t.div_(self.size) if hasattr(t, "div_") else t.__itruediv__(self.size)
        return t


class DataParallel(_Base):
    """Gradient synchronisation for data parallelism.

    Gradients are flattened into buckets of at most ``bucket_bytes`` (sized for launch
    latency and overlap, not link count — NVSwitch gives every peer full bandwidth)
    which live in symmetric memory, so each bucket is one zero-copy fused kernel.
    """

    def __init__(self, ctx, cuda_ctx=None, bucket_bytes: int = 64 << 20):
        super().__init__(ctx, cuda_ctx)
        self.bucket_bytes = bucket_bytes
        self._buckets = {}

    def broadcast_parameters(self, params: Iterable, root: int = 0):
        for p in params:
            t = p.data if hasattr(p, "data") else p
            if _is_cuda(t):
                self.cc.broadcast(t, root=root)
            else:
                H.broadcast(self.ctx, t, root=root)

    def _bucket(self, key, numel, dtype, device):
        b = self._buckets.get(key)
        if b is None or b.numel() < numel:
            if device.type == "cuda":
                b = self.cc.empty(numel, dtype)  # symmetric: zero-copy, NVLS-capable
            else:
                import torch

                b = torch.empty(numel, dtype=dtype)
            self._buckets[key] = b
        return b[:numel]

    def allreduce_gradients(self, params: Iterable, average: bool = True):
        import torch

        grads = [p.grad for p in params if getattr(p, "grad", None) is not None]
        if not grads:
            return
        groups, cur, cur_bytes = [], [], 0
        for g in grads:
            nbytes = g.numel() * g.element_size()
            if cur and (cur_bytes + nbytes > self.bucket_bytes or g.dtype != cur[0].dtype):
                groups.append(cur)
                cur, cur_bytes = [], 0
            cur.append(g)
            cur_bytes += nbytes
        if cur:
            groups.append(cur)
        for i, group in enumerate(groups):
            n = sum(g.numel() for g in group)
            flat = self._bucket((i, group[0].dtype), n, group[0].dtype, group[0].device)
            off = 0
            for g in group:
                flat[off:off + g.numel()].copy_(g.reshape(-1))
                off += g.numel()
            self._allreduce(flat, average=average)
            off = 0
            for g in group:
                g.copy_(flat[off:off + g.numel()].view_as(g))
                off += g.numel()


class GradientBucketer(_Base):
    """Gradient synchronisation that overlaps with the backward pass, without copies.

    Parameters are packed, in reverse order (the last layers finish their backward first), into
    flat buckets of at most ``bucket_bytes``. On CUDA a bucket is SYMMETRIC memory
    (``CudaContext.empty``: peer-mapped and, beyond two GPUs, bound to an NVSwitch multicast
    object) and every ``p.grad`` is a VIEW into its bucket, so autograd accumulates straight into
    the buffer the collective reads: no flatten / unflatten pass, and the allreduce is the zero-copy
    fused kernel (1/P average in its epilogue). A bucket is launched on a side stream as soon as
    the last of its gradients has been accumulated (``register_post_accumulate_grad_hook``), in
    bucket order on every rank; ``finish()`` makes the compute stream wait for the results.
    The reference has no counterpart (its consumers - ProcessGroupGloo + DDP's reducer - copy
    gradients into a bucket, stage it through pinned host memory and reduce on the CPU).

        bucketer = GradientBucketer(ctx, cuda_ctx, model.parameters())
        loss.backward(); bucketer.finish(); optimizer.step(); bucketer.zero_grad()
    """

    def __init__(self, ctx, cuda_ctx, params: Iterable, bucket_bytes: int = 64 << 20, average: bool = True):
        import torch

        super().__init__(ctx, cuda_ctx)
        self.average = average
        self.buckets = []
        self._next = 0
        self._hooks = []
        self._comm_stream = None
        # Ranks that share one GPU (threads-as-ranks tests) rendezvous on the host before every launch
        # (PeerContext::launchGuard) and share the process's single autograd thread: a hook that waits for
        # a peer's hook would wait for itself. There the buckets are launched from finish() instead.
        self._defer = cuda_ctx is not None and cuda_ctx.pc.ranks_on_my_device() > 1
        plist = [p for p in params if p.requires_grad]
        groups, cur, cur_bytes = [], [], 0
        for p in reversed(plist):
            nbytes = p.numel() * p.element_size()
            if cur and (cur_bytes + nbytes > bucket_bytes or p.dtype != cur[0].dtype or p.device != cur[0].device):
                groups.append(cur)
                cur, cur_bytes = [], 0
            cur.append(p)
            cur_bytes += nbytes
        if cur:
            groups.append(cur)
        for group in groups:
            # every view starts on a 16-byte boundary so the kernels stay vectorised
            align = max(1, 16 // group[0].element_size())
            offs, n = [], 0
            for p in group:
                offs.append(n)
                n += (p.numel() + align - 1) // align * align
            cuda = _is_cuda(group[0])
            if cuda:
                flat = self.cc.empty(n, group[0].dtype)
                if self._comm_stream is None:
                    from ..ops.cuda import new_stream  # dedicated: torch.cuda.Stream() comes from a shared pool

                    self._comm_stream = new_stream(group[0].device.index)
            else:
                flat = torch.empty(n, dtype=group[0].dtype)
            flat.zero_()
            b = {"flat": flat, "params": group, "offs": offs, "pending": len(group), "launched": False, "done": None,
                 "cuda": cuda}
            for p, off in zip(group, offs):
                p.grad = flat[off:off + p.numel()].view_as(p)
                self._hooks.append(p.register_post_accumulate_grad_hook(lambda q, b=b: self._ready(b, q)))
            self.buckets.append(b)

    def _view(self, b, p):
        off = b["offs"][[id(x) for x in b["params"]].index(id(p))]
        return b["flat"][off:off + p.numel()].view_as(p)

    def _ready(self, b, p):
        v = self._view(b, p)
        if p.grad is not None and p.grad.data_ptr() != v.data_ptr():
            # somebody replaced the gradient tensor (zero_grad(set_to_none=True), clip utilities that
            # rebind .grad): take the value and point .grad back into the bucket
            v.copy_(p.grad)
            p.grad = v
        b["pending"] -= 1
        if self._defer:
            return
        while self._next < len(self.buckets) and self.buckets[self._next]["pending"] == 0:
            self._launch(self.buckets[self._next])
            self._next += 1

    def _launch(self, b):
        if b["launched"]:
            return
        b["launched"] = True
        if b["cuda"]:
            import torch

            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            self._comm_stream.wait_event(ev)
            fused = self.average and b["flat"].is_floating_point()
            self.cc.allreduce(b["flat"], average=fused, stream=self._comm_stream)
            if self.average and not fused:
                with torch.cuda.stream(self._comm_stream):
                    b["flat"].div_(self.size)
            b["done"] = torch.cuda.Event()
            b["done"].record(self._comm_stream)
        else:
            self._allreduce(b["flat"], average=self.average)

    def finish(self):
        """After ``backward()``: launch what has not been launched (buckets with parameters that
        received no gradient this step) in order, and order the compute stream behind the results."""
        for b in self.buckets[self._next:]:
            self._launch(b)
        for b in self.buckets:
            if b["cuda"] and b["done"] is not None:
                import torch

                torch.cuda.current_stream().wait_event(b["done"])
            b["pending"], b["launched"], b["done"] = len(b["params"]), False, None
        self._next = 0

    def zero_grad(self):
        """Zero the buckets in place (keeps every ``p.grad`` a view into symmetric memory)."""
        for b in self.buckets:
            b["flat"].zero_()
            for p, off in zip(b["params"], b["offs"]):
                v = b["flat"][off:off + p.numel()].view_as(p)
                if p.grad is None or p.grad.data_ptr() != v.data_ptr():
                    p.grad = v

    def remove(self):
        for h in self._hooks:
            h.remove()
        self._hooks = []


class ZeroShard(_Base):
    """ZeRO / FSDP building blocks: each rank owns 1/P of a flat parameter vector."""

    def shard_range(self, numel: int):
        base, rem = divmod(numel, self.size)
        counts = [base + (1 if r < rem else 0) for r in range(self.size)]
        start = sum(counts[: self.rank])
        return start, counts[self.rank], counts

    def reduce_scatter_gradients(self, flat_grad, out_shard, average: bool = True):
        """``out_shard`` may have another dtype than ``flat_grad`` (e.g. bf16 gradients into an fp32
        shard): on CUDA the kernel converts (fp32 accumulation, 1/P on the accumulator, one
        rounding); on the host the gradient is converted with torch first."""
        _, _, counts = self.shard_range(flat_grad.numel())
        if _is_cuda(flat_grad):
            fused = average and flat_grad.is_floating_point()
            self.cc.reduce_scatter(out_shard, flat_grad, counts, scale=1.0 / self.size if fused else 1.0)
            if average and not fused:
                out_shard.div_(self.size)
        else:
            if getattr(flat_grad, "dtype", None) != getattr(out_shard, "dtype", None):
                flat_grad = flat_grad.to(out_shard.dtype)
            H.reduce_scatter(self.ctx, out_shard, flat_grad, counts)
            if average:
                out_shard.div_(self.size) if hasattr(out_shard, "div_") else None
        return out_shard

    def allgather_parameters(self, flat_param, shard):
        """``shard`` may have another dtype than ``flat_param`` (e.g. an fp32 master shard gathered
        into bf16 parameters): on CUDA each shard is converted once inside the kernel; on the host it
        is converted with torch first."""
        _, _, counts = self.shard_range(flat_param.numel())
        if _is_cuda(flat_param):
            self.cc.allgatherv(flat_param, shard, counts)
        else:
            if getattr(flat_param, "dtype", None) != getattr(shard, "dtype", None):
                shard = shard.to(flat_param.dtype)
            H.allgatherv(self.ctx, flat_param, counts, shard)
        return flat_param


class ZeroOptimizer(_Base):
    """ZeRO stage 1 on flat buffers: every rank keeps the optimizer state of 1/P of the parameters.

    Parameters and gradients are re-pointed into two flat buffers (symmetric memory on CUDA: the
    collectives read and write them in place). ``step()`` = reduce_scatter of the flat gradient
    (1/P average fused into the kernel) -> the wrapped torch optimizer updates this rank's shard
    only -> allgather of the updated shards back into the flat parameter buffer. Optimizer state
    (Adam moments, ...) exists for the shard only: 1/P of the memory of a replicated optimizer.

        zo = ZeroOptimizer(ctx, cuda_ctx, model.parameters(), torch.optim.AdamW, lr=1e-3)
        loss.backward(); zo.step(); zo.zero_grad()

    ``master_dtype`` (e.g. ``torch.float32`` for a bf16 / fp16 model) gives the optimizer master
    weights of that dtype: the shard and its gradient are ``master_dtype``, initialised from the
    upcast parameters, while the flat parameter and gradient buffers stay in the model dtype. On
    CUDA ``step()`` is then still two collective launches: a reduce_scatter that converts the
    gradients (fp32 accumulation, 1/P and one rounding inside the kernel) and an allgather that
    rounds the updated master shard once into the model dtype. ``None`` keeps one dtype.
    Exception: with a single rank both conversions run locally through the small-message (LL)
    kernel, one launch per ``GLB_CUDA_LL_MAX``-sized piece (16 KB by default), which is far slower
    than the same step without ``master_dtype`` for large models (see docs/cuda.md).
    """

    def __init__(self, ctx, cuda_ctx, params: Iterable, optimizer_cls, average: bool = True, master_dtype=None,
                 **optimizer_kwargs):
        import torch

        super().__init__(ctx, cuda_ctx)
        self.average = average
        self.params = [p for p in params if p.requires_grad]
        assert self.params, "no trainable parameters"
        dtype, device = self.params[0].dtype, self.params[0].device
        assert all(p.dtype == dtype and p.device == device for p in self.params), "one dtype / device per ZeroOptimizer"
        cuda = device.type == "cuda"
        align = max(1, 16 // self.params[0].element_size())
        offs, n = [], 0
        for p in self.params:
            offs.append(n)
            n += (p.numel() + align - 1) // align * align
        unit = align * self.size                       # every shard starts on a 16-byte boundary
        n = (n + unit - 1) // unit * unit
        alloc = (lambda k: self.cc.empty(k, dtype)) if cuda else (lambda k: torch.empty(k, dtype=dtype))
        self.flat_param, self.flat_grad = alloc(n), alloc(n)
        self.flat_param.zero_()
        self.flat_grad.zero_()
        with torch.no_grad():
            for p, off in zip(self.params, offs):
                self.flat_param[off:off + p.numel()].copy_(p.reshape(-1))
                p.data = self.flat_param[off:off + p.numel()].view_as(p)
                p.grad = self.flat_grad[off:off + p.numel()].view_as(p)
        self._offs = offs
        self.counts = [n // self.size] * self.size
        self.start = self.rank * (n // self.size)
        cnt = self.counts[self.rank]
        # the shard the optimizer owns: its own tensors (the collectives' inputs / outputs must not
        # alias the flat buffers they gather into / scatter from)
        # The padding above starts every shard on a 16-byte boundary of the model-dtype buffers, which
        # keeps the converting collectives on their vector path as well.
        src = self.flat_param[self.start:self.start + cnt].detach()
        self.master_dtype = master_dtype
        if master_dtype is None:
            self.shard = torch.nn.Parameter(src.clone())
        else:
            self.shard = torch.nn.Parameter(src.to(master_dtype, copy=True))
        self.shard.grad = torch.zeros_like(self.shard)
        self.optimizer = optimizer_cls([self.shard], **optimizer_kwargs)

    def step(self):
        import torch

        # a gradient tensor that was rebound (zero_grad(set_to_none=True)) is copied back into the flat buffer
        for p, off in zip(self.params, self._offs):
            v = self.flat_grad[off:off + p.numel()].view_as(p)
            if p.grad is not None and p.grad.data_ptr() != v.data_ptr():
                v.copy_(p.grad)
                p.grad = v
        ZeroShard(self.ctx, self.cc).reduce_scatter_gradients(self.flat_grad, self.shard.grad, average=self.average)
        self.optimizer.step()
        with torch.no_grad():
            ZeroShard(self.ctx, self.cc).allgather_parameters(self.flat_param, self.shard.data)

    def zero_grad(self):
        self.flat_grad.zero_()
        for p, off in zip(self.params, self._offs):
            v = self.flat_grad[off:off + p.numel()].view_as(p)
            if p.grad is None or p.grad.data_ptr() != v.data_ptr():
                p.grad = v

    def state_bytes(self) -> int:
        """Bytes of optimizer state held by this rank (for the 1/P claim)."""
        import torch

        return sum(v.numel() * v.element_size() for st in self.optimizer.state.values() for v in st.values()
                   if isinstance(v, torch.Tensor))


class TensorParallel(_Base):
    """Megatron tensor parallelism: row-parallel output is an allreduce of partial sums;
    column-parallel output is an allgather along the feature dimension.

    ``column_linear`` / ``row_linear`` build the two layers of a tensor-parallel MLP block with
    the collectives placed as autograd functions (Megatron's f / g operators): the forward of a
    column -> row pair costs ONE allreduce (after the row-parallel matmul), the backward one
    (before the column-parallel weight gradient)."""

    def row_parallel_output(self, partial):
        return self._allreduce(partial)

    def column_parallel_gather(self, local, out):
        if _is_cuda(local):
            self.cc.allgather(out, local)
        else:
            H.allgather(self.ctx, out, local)
        return out

    # ---- autograd-aware operators --------------------------------------------------------------
    def copy_to_region(self, x):
        """f: identity in the forward pass, allreduce of the gradient in the backward pass."""
        import torch

        tp = self

        class _F(torch.autograd.Function):
            @staticmethod
            def forward(ctx, inp):
                return inp.view_as(inp)

            @staticmethod
            def backward(ctx, grad):
                return tp._allreduce(grad.contiguous().clone())

        return _F.apply(x)

    def reduce_from_region(self, x):
        """g: allreduce in the forward pass, identity in the backward pass."""
        import torch

        tp = self

        class _G(torch.autograd.Function):
            @staticmethod
            def forward(ctx, inp):
                return tp._allreduce(inp.contiguous().clone())

            @staticmethod
            def backward(ctx, grad):
                return grad

        return _G.apply(x)

    def column_linear(self, in_features: int, out_features: int, bias: bool = True, device=None, dtype=None):
        return ColumnParallelLinear(self, in_features, out_features, bias, device, dtype)

    def row_linear(self, in_features: int, out_features: int, bias: bool = True, device=None, dtype=None):
        return RowParallelLinear(self, in_features, out_features, bias, device, dtype)


def _shard(n: int, size: int, rank: int):
    assert n % size == 0, f"{n} features do not split over {size} ranks"
    return n // size * rank, n // size * (rank + 1)


try:  # the layer classes need torch; everything else in this module does not
    import torch as _torch

    class ColumnParallelLinear(_torch.nn.Module):
        """y_local = x W_r^T + b_r with W split along the OUTPUT features (rank r holds rows
        [r, r+1) * out/P). The input is replicated; its gradient is summed over ranks (f)."""

        def __init__(self, tp: TensorParallel, in_features, out_features, bias=True, device=None, dtype=None):
            super().__init__()
            self.tp = tp
            self.lo, self.hi = _shard(out_features, tp.size, tp.rank)
            self.weight = _torch.nn.Parameter(_torch.empty(self.hi - self.lo, in_features, device=device, dtype=dtype))
            self.bias = _torch.nn.Parameter(_torch.zeros(self.hi - self.lo, device=device, dtype=dtype)) if bias else None
            _torch.nn.init.kaiming_uniform_(self.weight, a=5 ** 0.5)

        def load_full(self, weight, bias=None):
            with _torch.no_grad():
                self.weight.copy_(weight[self.lo:self.hi])
                if self.bias is not None and bias is not None:
                    self.bias.copy_(bias[self.lo:self.hi])

        def forward(self, x):
            return _torch.nn.functional.linear(self.tp.copy_to_region(x), self.weight, self.bias)

    class RowParallelLinear(_torch.nn.Module):
        """y = sum_r x_r W_r^T + b with W split along the INPUT features; the input arrives already
        split (the output of a ColumnParallelLinear); one allreduce of the partial products (g)."""

        def __init__(self, tp: TensorParallel, in_features, out_features, bias=True, device=None, dtype=None):
            super().__init__()
            self.tp = tp
            self.lo, self.hi = _shard(in_features, tp.size, tp.rank)
            self.weight = _torch.nn.Parameter(_torch.empty(out_features, self.hi - self.lo, device=device, dtype=dtype))
            self.bias = _torch.nn.Parameter(_torch.zeros(out_features, device=device, dtype=dtype)) if bias else None
            _torch.nn.init.kaiming_uniform_(self.weight, a=5 ** 0.5)

        def load_full(self, weight, bias=None):
            with _torch.no_grad():
                self.weight.copy_(weight[:, self.lo:self.hi])
                if self.bias is not None and bias is not None:
                    self.bias.copy_(bias)

        def forward(self, x_local):
            y = self.tp.reduce_from_region(_torch.nn.functional.linear(x_local, self.weight))
            return y if self.bias is None else y + self.bias
except ImportError:  # pragma: no cover
    ColumnParallelLinear = RowParallelLinear = None


class SequenceParallel(_Base):
    """Megatron sequence parallelism: reduce_scatter along the sequence going in,
    allgather coming out."""

    def scatter_reduce(self, full, shard):
        return ZeroShard(self.ctx, self.cc).reduce_scatter_gradients(full, shard, average=False)

    def gather(self, shard, full):
        return ZeroShard(self.ctx, self.cc).allgather_parameters(full, shard)


class MoEDispatcher(_Base):
    """Expert parallelism: tokens routed to experts living on other ranks.

    dispatch(): rows of ``tokens`` (already sorted by destination rank) are exchanged
    with alltoallv; the per-source receive counts come from a tiny alltoall of the
    send counts. combine() is the inverse exchange.
    """

    def exchange_counts(self, send_counts: Sequence[int]) -> List[int]:
        import numpy as np

        s = np.asarray(send_counts, dtype=np.int64)
        r = np.zeros_like(s)
        H.alltoall(self.ctx, r, s)
        return [int(x) for x in r]

    def dispatch(self, tokens, send_counts: Sequence[int], out, recv_counts: Optional[Sequence[int]] = None):
        if recv_counts is None:
            recv_counts = self.exchange_counts(send_counts)
        width = tokens.shape[-1] if tokens.dim() > 1 else 1
        sc = [c * width for c in send_counts]
        rc = [c * width for c in recv_counts]
        if _is_cuda(tokens):
            self.cc.alltoallv(out, rc, tokens, sc)
        else:
            H.alltoallv(self.ctx, out, rc, tokens, sc)
        return out, list(recv_counts)

    def combine(self, expert_out, recv_counts: Sequence[int], out, send_counts: Sequence[int]):
        # inverse of dispatch: what I received goes back to where it came from
        return self.dispatch(expert_out, recv_counts, out, send_counts)[0]


class UlyssesAttention(_Base):
    """DeepSpeed-Ulysses: [S/P, H, D] <-> [S, H/P, D] with one alltoall each way."""

    def seq_to_heads(self, x, out):
        if _is_cuda(x):
            self.cc.alltoall(out, x)
        else:
            H.alltoall(self.ctx, out, x)
        return out

    heads_to_seq = seq_to_heads

    def attention(self, q, k, v, causal: bool = False):
        """Full Ulysses attention: q / k / v are this rank's sequence shard [S/P, H, D]; one alltoall
        turns them into all positions of H/P heads ([S, H/P, D]), attention runs locally over the
        whole sequence, one alltoall brings the output back to [S/P, H, D]. On CUDA the exchange
        buffers are symmetric (zero-copy push kernels); three alltoalls in, one out."""
        import torch

        P, r = self.size, self.rank
        s_loc, Hh, D = q.shape
        assert Hh % P == 0, "heads must divide over the ranks"
        hp = Hh // P

        def alloc(n, like):
            return self.cc.empty(n, like.dtype) if _is_cuda(like) else torch.empty(n, dtype=like.dtype)

        def to_heads(x):      # [S/P, H, D] -> [S, H/P, D]
            send = x.view(s_loc, P, hp, D).transpose(0, 1).contiguous()      # block j = my positions of head group j
            out = alloc(send.numel(), x)
            self.seq_to_heads(send.view(-1), out)
            return out.view(P * s_loc, hp, D)                                # block i = rank i's positions, my heads

        def to_seq(y):        # [S, H/P, D] -> [S/P, H, D]
            send = y.contiguous()                                           # block i = positions of rank i
            out = alloc(send.numel(), y)
            self.seq_to_heads(send.view(-1), out)
            return out.view(P, s_loc, hp, D).transpose(0, 1).reshape(s_loc, Hh, D)

        qh, kh, vh = to_heads(q), to_heads(k), to_heads(v)
        o = torch.nn.functional.scaled_dot_product_attention(qh.transpose(0, 1), kh.transpose(0, 1), vh.transpose(0, 1),
                                                             is_causal=causal).transpose(0, 1)
        return to_seq(o)


class RingExchange(_Base):
    """Neighbour exchange for ring attention (KV rotation) and pipeline parallelism.

    CPU tensors go through UnboundBuffer send/recv. CUDA tensors: when ``recv`` is a symmetric /
    registered tensor (``kv_buffers``) the zero-copy kernel writes ``send`` straight into the right
    neighbour's copy of it (``CudaContext.exchange``: one pass, ~link rate); any other tensor goes
    through the fused send+recv kernel and its mailbox ring (``CudaContext.sendrecv``).
    """

    def kv_buffers(self, numel: int, dtype):
        """Two symmetric buffers to rotate between (every rank must call this in the same order)."""
        return self.cc.empty(numel, dtype), self.cc.empty(numel, dtype)

    def rotate(self, send, recv, step: int = 1):
        right, left = (self.rank + step) % self.size, (self.rank - step) % self.size
        if self.size == 1:
            recv.copy_(send)
            return recv
        if _is_cuda(send):
            self.cc.exchange(send, right, recv, left)   # falls back to sendrecv() for unregistered tensors
            return recv
        from ..types import describe

        sp, sn, sdt, _ = describe(send)
        rp, rn, _, _ = describe(recv)
        nbytes = send.numel() * send.element_size() if hasattr(send, "numel") else send.nbytes
        sb = self.ctx.create_unbound_buffer(sp, nbytes)
        rb = self.ctx.create_unbound_buffer(rp, nbytes)
        slot = _C.slot_build(0x7E, step)
        rb.recv(left, slot)
        sb.send(right, slot)
        rb.wait_recv()
        sb.wait_send()
        return recv

    def attention(self, q, k, v, causal: bool = False):
        """Ring attention (forward): rank r holds the queries and the K/V block of sequence shard r
        ([S/P, H, D] each); K/V blocks rotate once around the ring while every rank folds the block
        it currently holds into a running (max, sum, output) with the online-softmax recurrence, so
        no rank ever materialises more than two K/V blocks. The rotation of the NEXT block is
        posted before the current one is consumed (double buffer: on CUDA the two halves of a
        symmetric buffer, written by the neighbour's zero-copy ``exchange`` kernel on a side
        stream while the attention math runs). ``causal``: shard r attends to shards <= r.
        Returns [S/P, H, D] in q's dtype. The math is plain torch (fp32 accumulation)."""
        import torch

        P, r = self.size, self.rank
        scale = q.shape[-1] ** -0.5
        qf = q.float().transpose(0, 1)                                    # [H, Sq, D]
        m = torch.full(qf.shape[:2], float("-inf"), device=q.device)      # running max   [H, Sq]
        l = torch.zeros(qf.shape[:2], device=q.device)                    # running sum   [H, Sq]
        acc = torch.zeros_like(qf)                                        # running out   [H, Sq, D]
        kv = torch.stack([k, v]).contiguous()
        cuda = _is_cuda(kv)
        if cuda and P > 1:
            cur, nxt = self.kv_buffers(kv.numel(), kv.dtype)
            cur = cur.view_as(kv)
            nxt = nxt.view_as(kv)
            cur.copy_(kv)
            side = getattr(self, "_side", None)
            if side is None:
                from ..ops.cuda import new_stream

                side = self._side = new_stream(kv.device.index)
        else:
            cur, nxt = kv, torch.empty_like(kv)
        for step in range(P):
            src = (r - step) % P                                          # whose block `cur` is
            if step + 1 < P:                                              # post the next rotation first
                if cuda:
                    ready = torch.cuda.Event()
                    ready.record(torch.cuda.current_stream())
                    side.wait_event(ready)
                    self.cc.exchange(cur, (r + 1) % P, nxt, (r - 1) % P, stream=side)
                    landed = torch.cuda.Event()
                    landed.record(side)
                else:
                    self.rotate(cur, nxt)
            if not (causal and src > r):
                kf, vf = cur[0].float().transpose(0, 1), cur[1].float().transpose(0, 1)   # [H, Sk, D]
                s = torch.matmul(qf, kf.transpose(1, 2)) * scale                          # [H, Sq, Sk]
                if causal and src == r:
                    sq, sk = s.shape[-2:]
                    s = s.masked_fill(torch.ones(sq, sk, dtype=torch.bool, device=s.device).triu(1), float("-inf"))
                m_new = torch.maximum(m, s.amax(dim=-1))
                p = torch.exp(s - m_new.unsqueeze(-1))
                alpha = torch.exp(m - m_new)
                l = l * alpha + p.sum(dim=-1)
                acc = acc * alpha.unsqueeze(-1) + torch.matmul(p, vf)
                m = m_new
            if step + 1 < P:
                if cuda:
                    torch.cuda.current_stream().wait_event(landed)
                cur, nxt = nxt, cur
        return (acc / l.unsqueeze(-1)).transpose(0, 1).to(q.dtype)


class PipelineParallel(_Base):
    """Pipeline parallelism (GPipe schedule): rank r holds stage r of the model; micro-batches flow
    forward through point-to-point sends of the activations and backward through sends of their
    gradients. All forwards run first, then all backwards in reverse micro-batch order, so every
    stage keeps at most ``len(microbatches)`` activations alive and parameter gradients accumulate
    over the micro-batches exactly as in one big batch.

    CPU tensors move through unbound-buffer send / recv; CUDA tensors through the NVLink
    point-to-point kernels (``CudaContext.send`` / ``recv``: the receiver drains a mailbox ring
    inside its own pool while the sender streams into it, both on the current stream).
    Activation shapes must be the same for every micro-batch (``out_shape`` of the previous stage).
    """

    _TAG_FWD, _TAG_BWD = 0x50, 0x51

    def _send(self, t, dst, tag, seq):
        if _is_cuda(t):
            self.cc.send(t.contiguous(), dst)
            return
        t = t.contiguous()
        b = self.ctx.create_unbound_buffer(t.data_ptr(), t.numel() * t.element_size())
        b.send(dst, _C.slot_build(tag, seq))
        b.wait_send()

    def _recv(self, t, src, tag, seq):
        if _is_cuda(t):
            self.cc.recv(t, src)
            return t
        b = self.ctx.create_unbound_buffer(t.data_ptr(), t.numel() * t.element_size())
        b.recv(src, _C.slot_build(tag, seq))
        b.wait_recv()
        return t

    def run(self, stage, microbatches: Sequence, in_shape=None, loss_fn=None, targets: Optional[Sequence] = None,
            dtype=None, device=None):
        """One training step. ``stage``: this rank's module. ``microbatches``: the inputs (first stage only,
        elsewhere just their count matters). ``in_shape``: shape of the activation this stage receives (all but
        the first stage). ``loss_fn(output, target)`` and ``targets`` on the last stage. Returns the list of
        micro-batch losses on the last stage, ``None`` elsewhere; parameter gradients are left in ``.grad``
        (summed over micro-batches; scale the loss by 1/len(microbatches) for a mean)."""
        import torch

        first, last = self.rank == 0, self.rank == self.size - 1
        n = len(microbatches)
        inputs, outputs, losses = [], [], []
        for i in range(n):
            if first:
                x = microbatches[i]
            else:
                x = self._recv(torch.empty(in_shape, dtype=dtype, device=device), self.rank - 1, self._TAG_FWD, i)
                x.requires_grad_(True)
            y = stage(x)
            inputs.append(x)
            if last:
                loss = loss_fn(y, targets[i])
                losses.append(loss)
                outputs.append(loss)
            else:
                outputs.append(y)
                self._send(y.detach(), self.rank + 1, self._TAG_FWD, i)
        for i in reversed(range(n)):
            if last:
                outputs[i].backward()
            else:
                g = self._recv(torch.empty_like(outputs[i]), self.rank + 1, self._TAG_BWD, i)
                outputs[i].backward(g)
            if not first:
                self._send(inputs[i].grad, self.rank - 1, self._TAG_BWD, i)
        return [float(l.detach()) for l in losses] if last else None
