"""Bit-exact numerics of the converting reduce_scatter and allgather(v) (f32 <-> f16 / bf16).

Threads act as ranks on cuda:0 at P = 1, 2, 3, 4 and 8 and compare raw output bits with
``reduction_oracle``: reduce_scatter must equal ``ro.expected(inputs, op, scale, src, out=dst)``
on the rank's share (fp32 accumulation, scale, one rounding), allgather must equal the one
conversion of every block. A rank never raises on a mismatch (its peers would be left waiting
inside a collective); it collects failures and the main thread reports them.
"""
import os
import subprocess
import sys
import tempfile
import zlib

import numpy as np
import pytest

import mixed_precision_common as mp
import reduction_oracle as ro

BUF_BYTES = 4 << 20
RS_KINDS = ("plain", "plain+1", "registered", "symmetric")
AG_KINDS = ("plain", "registered", "symmetric")


def _torch(name):
    import torch

    return {"f16": torch.float16, "bf16": torch.bfloat16, "f32": torch.float32}[name]


def _upload(dst, bits):
    import torch

    signed = {2: np.int16, 4: np.int32}[bits.dtype.itemsize]
    raw = {2: torch.int16, 4: torch.int32}[dst.element_size()]
    dst.view(raw).copy_(torch.from_numpy(np.ascontiguousarray(bits).view(signed)))


def _download(t, name):
    import torch

    raw = {2: torch.int16, 4: torch.int32}[t.element_size()]
    return t.detach().view(raw).cpu().numpy().view(ro.dtype(name).bits)


class _Bufs:
    def __init__(self, cc):
        import torch

        self.plain = torch.empty(BUF_BYTES, dtype=torch.uint8, device="cuda")
        self.reg = torch.empty(BUF_BYTES, dtype=torch.uint8, device="cuda")
        cc.register(self.reg)
        self.sym = cc.empty(BUF_BYTES, torch.uint8)

    def view(self, kind, name, n):
        es = np.dtype(ro.dtype(name).bits).itemsize
        base = {"plain": self.plain, "registered": self.reg, "symmetric": self.sym}[kind.split("+")[0]]
        off = es if kind.endswith("+1") else 0
        assert off + n * es <= BUF_BYTES
        return base[off:off + n * es].view(_torch(name))


def _gop(op):
    import gloo_b200 as gb

    return {ro.SUM: gb.ReduceOp.SUM, ro.PRODUCT: gb.ReduceOp.PRODUCT, ro.MIN: gb.ReduceOp.MIN,
            ro.MAX: gb.ReduceOp.MAX}[op]


def _context(ctx):
    from gloo_b200.ops import cuda as gcu

    cc = gcu.CudaContext(ctx, 0, stage_bytes=8 << 20)
    cc.set_timeout(60000)
    return cc


def _run_ranks(P, fn):
    import gloo_b200 as gb

    res = gb.spawn_threads(P, fn, cuda_device=0, timeout_ms=120000)
    failures = [f"rank {r}: {m}" for r, out in enumerate(res) for m in out["fail"]]
    assert not failures, f"{len(failures)} failures:\n" + "\n".join(failures[:40])
    return res


def _rs_tables(P):
    """(label, counts): LL-sized equal shares, even shares, the default split of an uneven
    count, and skewed shares whose offsets are not 16-byte aligned."""
    skew = [1, 4103, 17, 60001, 3, 999, 5, 20001][:P]
    return [("ll", [100] * P), ("even", [20000] * P), ("uneven", None), ("skewed", skew)]


def _split(n, P):
    base, rem = divmod(n, P)
    return [base + (1 if r < rem else 0) for r in range(P)]


class _Data:
    def __init__(self, P, n):
        self.P, self.n = P, n
        self._in, self._out = {}, {}

    def inputs(self, name, op):
        key = (name, op)
        if key not in self._in:
            vals = ro.exact_inputs(self.P, self.n, name, seed=zlib.crc32(f"mp/{name}/{op}/{self.P}".encode()), op=op)
            self._in[key] = (vals, [ro.to_bits(v, name) for v in vals])
        return self._in[key]

    def expected(self, src, dst, op, scale):
        key = (src, dst, op, scale)
        if key not in self._out:
            self._out[key] = ro.expected(self.inputs(src, op)[0], op, scale, src, out=dst)
        return self._out[key]


@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 2, 3, 4, 8])
def test_reduce_scatter_cast_bitwise(P):
    """4 pairs x SUM / PRODUCT / MIN / MAX x scale 1, 1/P, 0.3 x share tables x input kinds."""

    def fn(ctx):
        import torch

        cc = _context(ctx)
        bufs = _Bufs(cc)
        data = _Data(P, 160003)
        fail, ran = [], 0
        for src, dst in mp.PAIRS:
            for op in ro.OPS:
                for scale in (1.0, 1.0 / P, 0.3):
                    for label, counts in _rs_tables(P):
                        counts = _split(100003, P) if counts is None else counts
                        n = sum(counts)
                        off = sum(counts[:ctx.rank])
                        want = data.expected(src, dst, op, scale)[off:off + counts[ctx.rank]]
                        for kind in RS_KINDS:
                            inp = bufs.view(kind, src, n)
                            _upload(inp, data.inputs(src, op)[1][ctx.rank][:n])
                            # "+1": the output is one element off 16-byte alignment too
                            extra = 1 if kind.endswith("+1") else 0
                            out = torch.empty(counts[ctx.rank] + extra, dtype=_torch(dst), device="cuda")[extra:]
                            cc.reduce_scatter(out, inp, counts=counts, op=_gop(op), scale=scale)
                            cc.synchronize()
                            msg = ro.mismatch(_download(out, dst), want, dst)
                            ran += 1
                            if msg:
                                fail.append(f"reduce_scatter {src}->{dst} {op} scale={scale:.4g} {label} {kind}: {msg}")
        cc.pc.host_barrier()
        return {"fail": fail, "ran": ran}

    res = _run_ranks(P, fn)
    assert res[0]["ran"] == 4 * 4 * 3 * 4 * len(RS_KINDS)


def _ag_tables(P):
    """(label, counts): equal blocks (allgather) of several sizes, then uneven counts whose
    offsets are not 16-byte aligned, one of them empty."""
    tables = [(f"allgather{n}", [n] * P) for n in (1, 7, 4103, 65537)]
    tables.append(("v-uneven", [4103 + 3 * r for r in range(P)]))
    tables.append(("v-empty", [0 if r == P // 2 else 1001 + 5 * r for r in range(P)]))
    return tables


@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 2, 3, 4, 8])
def test_allgather_cast_bitwise(P):
    """4 pairs x plain / registered / symmetric outputs x equal and uneven counts, random bits
    (Inf, NaN, subnormals, f16 overflow) and exact ties: each block is converted once."""

    def fn(ctx):
        import torch

        cc = _context(ctx)
        bufs = _Bufs(cc)
        fail, ran = [], 0
        for src, dst in mp.PAIRS:
            for label, counts in _ag_tables(P):
                blocks = []
                for r in range(P):
                    b = mp.random_bits(counts[r], src, seed=zlib.crc32(f"ag/{src}/{label}/{P}/{r}".encode()))
                    if src == "f32" and counts[r] > 64:
                        b[:64] = mp.tie_bits(64, dst, seed=r)
                    blocks.append(b)
                want = mp.convert_bits(np.concatenate(blocks), src, dst)
                inp = torch.empty(counts[ctx.rank], dtype=_torch(src), device="cuda")
                _upload(inp, blocks[ctx.rank])
                for kind in AG_KINDS:
                    out = bufs.view(kind, dst, sum(counts))
                    if label.startswith("allgather"):
                        cc.allgather(out, inp)
                    else:
                        cc.allgatherv(out, inp, counts)
                    cc.synchronize()
                    msg = ro.mismatch(_download(out, dst), want, dst)
                    ran += 1
                    if msg:
                        fail.append(f"allgather {src}->{dst} {label} {kind}: {msg}")
        cc.pc.host_barrier()
        return {"fail": fail, "ran": ran}

    res = _run_ranks(P, fn)
    assert res[0]["ran"] == 4 * len(_ag_tables(P)) * len(AG_KINDS)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 2, 4])
def test_edge_values_and_checks(P):
    """Signed zeros, Inf, NaN, f16 overflow and subnormals through both calls; mismatched
    lengths raise ValueError and unsupported pairs TypeError without launching anything."""

    def fn(ctx):
        import torch

        import gloo_b200 as gb

        cc = _context(ctx)
        fail, ran = [], 0
        for src, dst in mp.PAIRS:
            e = mp.edge_values(src)
            vals = [e] * P  # every column holds one edge value on every rank
            n = len(e)
            for scale in (1.0, 0.3):
                with np.errstate(all="ignore"):
                    want = ro.expected([np.tile(v, P) for v in vals], ro.SUM, scale, src, out=dst)
                inp = torch.empty(n * P, dtype=_torch(src), device="cuda")
                _upload(inp, ro.to_bits(np.tile(vals[ctx.rank], P), src))
                out = torch.empty(n, dtype=_torch(dst), device="cuda")
                cc.reduce_scatter(out, inp, scale=scale)
                cc.synchronize()
                msg = ro.mismatch(_download(out, dst), want[ctx.rank * n:(ctx.rank + 1) * n], dst)
                ran += 1
                if msg:
                    fail.append(f"edge reduce_scatter {src}->{dst} scale={scale}: {msg}")
            mine = torch.empty(n, dtype=_torch(src), device="cuda")
            _upload(mine, ro.to_bits(e, src))
            g = torch.empty(n * P, dtype=_torch(dst), device="cuda")
            cc.allgather(g, mine)
            cc.synchronize()
            msg = ro.mismatch(_download(g, dst), np.tile(mp.convert_bits(ro.to_bits(e, src), src, dst), P), dst)
            ran += 1
            if msg:
                fail.append(f"edge allgather {src}->{dst}: {msg}")
        # the counter is shared by every rank in this process: wait until no peer can still be
        # finishing a launch before reading it (the refused calls below launch nothing)
        cc.pc.host_barrier()
        before = gb._C.cuda.launch_count()
        bad = [
            (ValueError, lambda: cc.reduce_scatter(torch.empty(7, dtype=torch.bfloat16, device="cuda"),
                                                   torch.empty(8 * P, device="cuda"))),
            (ValueError, lambda: cc.reduce_scatter(torch.empty(8, device="cuda"), torch.empty(8 * P - 1, device="cuda"),
                                                   counts=[8] * P)),
            (ValueError, lambda: cc.allgather(torch.empty(8 * P - 1, dtype=torch.bfloat16, device="cuda"),
                                              torch.empty(8, device="cuda"))),
            (TypeError, lambda: cc.reduce_scatter(torch.empty(8, dtype=torch.bfloat16, device="cuda"),
                                                  torch.empty(8 * P, dtype=torch.float16, device="cuda"))),
            (TypeError, lambda: cc.allgather(torch.empty(8 * P, dtype=torch.float64, device="cuda"),
                                             torch.empty(8, device="cuda"))),
        ]
        for exc, call in bad:
            try:
                call()
                fail.append(f"{exc.__name__} not raised")
            except exc:
                pass
        if gb._C.cuda.launch_count() != before:
            fail.append("a refused call launched a kernel")
        cc.pc.host_barrier()
        return {"fail": fail, "ran": ran}

    _run_ranks(P, fn)


@pytest.mark.gpu
def test_zero_optimizer_master_fp32_on_gpu():
    """Threads as two ranks on one GPU: the fp32 master shard matches the emulation and the bf16
    parameters are within one bf16 ulp of its downcast; a step is two collective launches."""
    import torch

    import gloo_b200 as gb
    from gloo_b200.parallel import ZeroOptimizer

    P, steps = 2, 3

    def fn(ctx):
        cc = _context(ctx)
        g = torch.Generator().manual_seed(0)
        m = torch.nn.Linear(301, 97).to(torch.bfloat16)
        with torch.no_grad():
            for p in m.parameters():
                p.copy_(torch.randn(p.shape, generator=g))
        m = m.cuda()
        zo = ZeroOptimizer(ctx, cc, m.parameters(), torch.optim.AdamW, master_dtype=torch.float32, lr=1e-2)
        p0 = zo.flat_param.detach().cpu().clone()
        launches = []
        for s in range(steps):
            gg = torch.Generator().manual_seed(1000 * s + ctx.rank)
            for p in m.parameters():
                p.grad.copy_(torch.randn(p.shape, generator=gg).to(torch.bfloat16))
            cc.pc.host_barrier()
            # ranks that share a GPU meet on the host before every launch, so both read the
            # counter before either launches; it counts the launches of both ranks
            before = gb._C.cuda.launch_count()
            zo.step()
            cc.synchronize()
            cc.pc.host_barrier()
            launches.append(gb._C.cuda.launch_count() - before)
            zo.zero_grad()
        return {"fail": [], "p0": p0, "shard": zo.shard.detach().cpu(), "start": zo.start, "offs": zo._offs,
                "flat": zo.flat_param.detach().cpu(), "launches": launches}

    res = _run_ranks(P, fn)
    n = res[0]["flat"].numel()
    grads = []
    m = torch.nn.Linear(301, 97)
    shapes = [p.shape for p in m.parameters()]
    for s in range(steps):
        per_rank = []
        for r in range(P):
            gg = torch.Generator().manual_seed(1000 * s + r)
            flat = torch.zeros(n, dtype=torch.bfloat16)
            for shp, off in zip(shapes, res[0]["offs"]):
                k = int(np.prod(shp))
                flat[off:off + k] = torch.randn(shp, generator=gg).to(torch.bfloat16).reshape(-1)
            per_rank.append(flat)
        grads.append(per_rank)
    master, bf16 = mp.zero_emulation(grads, res[0]["p0"], steps)
    for r in res:
        assert r["launches"] == [2 * P] * steps, r["launches"]  # one reduce_scatter + one allgather per rank
        torch.testing.assert_close(r["shard"], master[r["start"]:r["start"] + r["shard"].numel()], rtol=1e-6, atol=1e-7)
        ulps = (r["flat"].view(torch.int16).int() - bf16.view(torch.int16).int()).abs()
        assert int(ulps.max()) <= 1


# ---- one process per GPU ------------------------------------------------------------------------------

WORKER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cuda_mixed_precision_worker.py")


def _gpu_count():
    try:
        import torch

        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.multigpu
@pytest.mark.skipif(_gpu_count() < 2, reason="needs >= 2 GPUs")
def test_mixed_precision_one_process_per_gpu():
    n = _gpu_count()
    size = 8 if n >= 8 else (4 if n >= 4 else 2)
    d = tempfile.mkdtemp(prefix="glb_mixed_mp_")
    procs = [subprocess.Popen([sys.executable, WORKER, d, str(r), str(size)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(size)]
    outs = []
    for p in procs:
        try:
            o, _ = p.communicate(timeout=600)
        except subprocess.TimeoutExpired:
            p.kill()
            o, _ = p.communicate()
        outs.append(o)
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"WORKER {r} OK" in o, f"rank {r} failed:\n{o[-4000:]}"
    print(outs[0][-2000:])
