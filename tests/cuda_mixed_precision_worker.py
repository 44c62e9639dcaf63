"""One process per GPU: the converting reduce_scatter (all four ops; plain, registered and
symmetric inputs) and allgather(v) (plain, registered and symmetric outputs) over real NVLink,
bit for bit against ``reduction_oracle``, and ``ZeroOptimizer(master_dtype=torch.float32)`` on a bf16
model against the single-process emulation.
usage: cuda_mixed_precision_worker.py STORE_DIR RANK SIZE"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import gloo_b200 as gb  # noqa: E402
import mixed_precision_common as mp  # noqa: E402
import reduction_oracle as ro  # noqa: E402
from gloo_b200.ops import cuda as gcu  # noqa: E402
from gloo_b200.parallel import ZeroOptimizer  # noqa: E402

TORCH = {"f16": torch.float16, "bf16": torch.bfloat16, "f32": torch.float32}
RAW = {2: torch.int16, 4: torch.int32}
SIGNED = {2: np.int16, 4: np.int32}


def upload(dst, bits):
    dst.view(RAW[dst.element_size()]).copy_(torch.from_numpy(np.ascontiguousarray(bits).view(SIGNED[bits.dtype.itemsize])))


def download(t, name):
    return t.view(RAW[t.element_size()]).cpu().numpy().view(ro.dtype(name).bits)


def zero_check(ctx, cc, rank, size, fail):
    steps = 3
    g = torch.Generator().manual_seed(0)
    m = torch.nn.Sequential(torch.nn.Linear(1024, 1031), torch.nn.Linear(1031, 77)).to(torch.bfloat16)
    with torch.no_grad():
        for p in m.parameters():
            p.copy_(torch.randn(p.shape, generator=g))
    m = m.cuda()
    zo = ZeroOptimizer(ctx, cc, m.parameters(), torch.optim.AdamW, master_dtype=torch.float32, lr=1e-2)
    p0 = zo.flat_param.detach().cpu().clone()
    n = p0.numel()
    shapes = [p.shape for p in m.parameters()]
    for s in range(steps):
        gg = torch.Generator().manual_seed(1000 * s + rank)
        for p in m.parameters():
            p.grad.copy_(torch.randn(p.shape, generator=gg).to(torch.bfloat16))
        before = gb._C.cuda.launch_count()
        zo.step()
        if gb._C.cuda.launch_count() - before != 2:
            fail.append(f"ZeroOptimizer step launched {gb._C.cuda.launch_count() - before} kernels, want 2")
        zo.zero_grad()
    cc.synchronize()
    grads = []
    for s in range(steps):
        per_rank = []
        for r in range(size):
            gg = torch.Generator().manual_seed(1000 * s + r)
            flat = torch.zeros(n, dtype=torch.bfloat16)
            for shp, off in zip(shapes, zo._offs):
                k = int(np.prod(shp))
                flat[off:off + k] = torch.randn(shp, generator=gg).to(torch.bfloat16).reshape(-1)
            per_rank.append(flat)
        grads.append(per_rank)
    master, bf16 = mp.zero_emulation(grads, p0, steps)
    shard = zo.shard.detach().cpu()
    try:
        torch.testing.assert_close(shard, master[zo.start:zo.start + shard.numel()], rtol=1e-6, atol=1e-7)
    except AssertionError as e:
        fail.append(f"ZeroOptimizer master shard: {e}")
    ulps = (zo.flat_param.detach().cpu().view(torch.int16).int() - bf16.view(torch.int16).int()).abs()
    if int(ulps.max()) > 1:
        fail.append(f"ZeroOptimizer bf16 parameters differ by {int(ulps.max())} ulp")


def main():
    store_dir, rank, size = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    ctx = gb.init_context(rank, size, path=store_dir, timeout_ms=60000)
    cc = gcu.CudaContext(ctx, dev, stage_bytes=64 << 20)
    cc.set_timeout(60000)
    fail, ran = [], 0
    tables = [("even", [1 << 19] * size), ("uneven", [3_000_001 // size + (1 if r < 3_000_001 % size else 0)
                                                      for r in range(size)]),
              ("skewed", [1, 4103, 17, 60001, 3, 999, 5, 20001][:size])]
    nmax = max(sum(c) for _, c in tables)
    cases = [(ro.SUM, (1.0, 1.0 / size, 0.3))] + [(op, (1.0, 0.3)) for op in (ro.PRODUCT, ro.MIN, ro.MAX)]
    gop = {ro.SUM: gb.ReduceOp.SUM, ro.PRODUCT: gb.ReduceOp.PRODUCT, ro.MIN: gb.ReduceOp.MIN, ro.MAX: gb.ReduceOp.MAX}
    for src, dst in mp.PAIRS:
        sym = cc.empty(nmax + 8, TORCH[src])
        reg = torch.empty(nmax + 8, dtype=TORCH[src], device="cuda")
        cc.register(reg)
        for op, scales in cases:
            vals = ro.exact_inputs(size, nmax, src, seed=17 + len(src) + 100 * ro.OPS.index(op), op=op)
            mine = ro.to_bits(vals[rank], src)
            for label, counts in tables:
                n = sum(counts)
                off = sum(counts[:rank])
                share = [v[off:off + counts[rank]] for v in vals]  # the model is elementwise: only my share
                for scale in scales:
                    want = ro.expected(share, op, scale, src, out=dst)
                    for kind in ("plain", "registered", "symmetric", "symmetric+1"):
                        base = {"registered": reg, "symmetric": sym, "symmetric+1": sym[1:]}.get(kind)
                        inp = torch.empty(n, dtype=TORCH[src], device="cuda") if base is None else base[:n]
                        upload(inp, mine[:n])
                        out = torch.empty(counts[rank], dtype=TORCH[dst], device="cuda")
                        cc.reduce_scatter(out, inp, counts=counts, op=gop[op], scale=scale)
                        cc.synchronize()
                        msg = ro.mismatch(download(out, dst), want, dst)
                        ran += 1
                        if msg:
                            fail.append(f"reduce_scatter {src}->{dst} {op} {label} {kind} scale={scale:.4g}: {msg}")
            del vals, mine
        # allgather(v): random bits, every block converted once
        for label, counts in (("even", [1 << 20] * size), ("uneven", [4103 + 3 * r for r in range(size)])):
            blocks = [mp.random_bits(counts[r], src, seed=100 * r + len(label)) for r in range(size)]
            want = mp.convert_bits(np.concatenate(blocks), src, dst)
            inp = torch.empty(counts[rank], dtype=TORCH[src], device="cuda")
            upload(inp, blocks[rank])
            for kind in ("plain", "registered", "symmetric"):
                if kind == "plain":
                    out = torch.empty(sum(counts), dtype=TORCH[dst], device="cuda")
                elif kind == "registered":
                    out = torch.empty(sum(counts), dtype=TORCH[dst], device="cuda")
                    cc.register(out)
                else:
                    out = cc.empty(sum(counts), TORCH[dst])
                cc.allgatherv(out, inp, counts)
                cc.synchronize()
                msg = ro.mismatch(download(out, dst), want, dst)
                ran += 1
                if msg:
                    fail.append(f"allgather {src}->{dst} {label} {kind}: {msg}")
        del sym
    zero_check(ctx, cc, rank, size, fail)
    cc.pc.host_barrier()
    for f in fail:
        print("FAIL", f, flush=True)
    print(f"RAN {ran}", flush=True)
    if not fail:
        print(f"WORKER {rank} OK", flush=True)


if __name__ == "__main__":
    main()
