"""One process per GPU: bit-exact numerics of the kernels that threads on one GPU cannot reach
(NVLS, the NVLS + peer-to-peer hybrid, the pipelined allreduce over a multicast staging
pool, the NVLS cast epilogue), against ``reduction_oracle``.
usage: cuda_numerics_worker.py STORE_DIR RANK SIZE"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import gloo_b200 as gb  # noqa: E402
import reduction_oracle as ro  # noqa: E402
from gloo_b200.ops import cuda as gcu  # noqa: E402

TORCH = {"f16": torch.float16, "bf16": torch.bfloat16, "f32": torch.float32}
RAW = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}
SIGNED = {2: np.int16, 4: np.int32}


def upload(dst, bits):
    dst.view(RAW[dst.element_size()]).copy_(torch.from_numpy(np.ascontiguousarray(bits).view(SIGNED[bits.dtype.itemsize])))


def download(t, name):
    return t.view(RAW[t.element_size()]).cpu().numpy().view(ro.dtype(name).bits)


def check_nvls(got, vals, scale, name, tail_start):
    """multimem.ld_reduce returns the dtype, so a 16-bit NVLS result with a non-dyadic scale
    is rounded twice (round(round(sum) * scale)) on the packs the switch reduced; packs
    reduced peer to peer and the sub-pack tail round once. Each element must match one of the
    two models exactly; the tail (which never goes through the switch) must round once."""
    once = ro.expected(vals, ro.SUM, scale, name)
    twice = ro.expected(vals, ro.SUM, scale, name, nvls=True)
    if ro.mismatch(got, once, name) is None or ro.mismatch(got, twice, name) is None:
        return None
    either = np.where(got == twice, twice, once)
    msg = ro.mismatch(got, either, name)
    if msg is None:
        msg = ro.mismatch(got[tail_start:], once[tail_start:], name)
    return msg


def main():
    store_dir, rank, size = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
    dev = rank % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    ctx = gb.init_context(rank, size, path=store_dir, timeout_ms=60000)
    cc = gcu.CudaContext(ctx, dev, stage_bytes=64 << 20)
    cc.set_timeout(60000)
    fail, ran = [], 0
    counts = (1, 7, 8 * size + 1, 4103, 65537, 1 << 20, 3_000_001)
    nmax = max(counts)

    def inputs(name, seed):
        vals = ro.exact_inputs(size, nmax, name, seed=seed)
        return vals, ro.to_bits(vals[rank], name)

    algos = ["two_shot", "auto"]
    if cc.nvls_available():
        algos += ["nvls"] + (["hybrid"] if size in (2, 4, 8) else [])
    for name in ("f32", "f16", "bf16"):
        vals, mine = inputs(name, 100 + len(name))
        sym = cc.empty(nmax + 8, TORCH[name])
        for algo in algos + ["pipelined"]:
            for scale in (1.0, 1.0 / size, 0.3):
                for n in counts:
                    t = torch.empty(n, dtype=TORCH[name], device="cuda") if algo == "pipelined" else sym[:n]
                    upload(t, mine[:n])
                    kw = {"blocks": 48, "unroll": 16, "tile": 300} if algo == "hybrid" else {}
                    cc.allreduce(t, algo=algo, scale=scale, **kw)
                    cc.synchronize()
                    got = download(t, name)
                    sub = [v[:n] for v in vals]
                    if algo in ("nvls", "hybrid", "auto", "pipelined") and name != "f32":
                        msg = check_nvls(got, sub, scale, name, n // 8 * 8)
                    else:
                        msg = ro.mismatch(got, ro.expected(sub, ro.SUM, scale, name), name)
                    ran += 1
                    if msg:
                        fail.append(f"{algo} {name} n={n} scale={scale:.4g}: {msg}")
    # cast epilogue: f32 -> 16-bit through multimem.ld_reduce (f32 accumulate: rounds once)
    vals, mine = inputs("f32", 7)
    for out_name in ("bf16", "f16"):
        for n in (4103, 1 << 20):
            src = cc.empty(n, torch.float32)
            dst = cc.empty(n, TORCH[out_name])
            upload(src, mine[:n])
            for scale in (1.0, 0.3):
                cc.allreduce(src, out=dst, scale=scale)
                cc.synchronize()
                want = ro.expected([v[:n] for v in vals], ro.SUM, scale, "f32", out=out_name)
                msg = ro.mismatch(download(dst, out_name), want, out_name)
                ran += 1
                if msg:
                    fail.append(f"cast f32->{out_name} n={n} scale={scale}: {msg}")
    cc.pc.host_barrier()
    for f in fail:
        print("FAIL", f, flush=True)
    print(f"RAN {ran} nvls={cc.nvls_available()}", flush=True)
    if not fail:
        print(f"WORKER {rank} OK", flush=True)


if __name__ == "__main__":
    main()
