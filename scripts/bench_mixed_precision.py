"""Mixed-precision sharded-training collectives, one process per GPU.

    python -m torch.distributed.run --nproc_per_node=8 scripts/bench_mixed_precision.py [--iters 20]

For bf16 parameter vectors of 4 MB to 1 GB it times, with CUDA events and the maximum over ranks:
  (a) reduce_scatter bf16 -> f32: the converting kernel, against upcast + f32 reduce_scatter and
      against a plain bf16 reduce_scatter;
  (b) allgather f32 -> bf16: the converting kernel, against f32 allgather + downcast and against
      downcast + bf16 allgather;
  (c) ZeroOptimizer.step() (AdamW) on a bf16 model larger than L2, with master_dtype=torch.float32
      and without.
Inputs are symmetric buffers (zero-copy) and the outputs plain tensors, as ZeroOptimizer uses
them. L2 is not flushed between passes: rows whose bf16 vector fits the 126 MB L2 of a B200 (4 to 64 MB
at the default sizes) measure largely L2-resident traffic; the JSON marks them with "l2_resident": true. Prints one JSON line (rank 0) that includes
the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import gloo_b200 as gb  # noqa: E402
from gloo_b200.ops import cuda as gcu  # noqa: E402
from gloo_b200.ops import host as H  # noqa: E402
from gloo_b200.parallel import ZeroOptimizer  # noqa: E402

SIZES_MB = (4, 16, 64, 256, 1024)
L2_MB = 126  # B200; not flushed between passes


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        name, power = [x.strip() for x in q.strip().split(",")[:2]]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # report what happened instead of guessing
        return {"gpu": torch.cuda.get_device_name(), "power_limit": f"unavailable ({type(e).__name__})"}


def timed(fn, cc, iters, warmup):
    """Mean time per call in microseconds, the maximum over ranks."""
    for _ in range(warmup):
        fn()
    cc.synchronize()
    cc.barrier()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    end.synchronize()
    us = torch.tensor([start.elapsed_time(end) * 1000.0 / iters], dtype=torch.float64)
    H.allreduce(cc.ctx, us.numpy(), op=gb.ReduceOp.MAX)
    return round(float(us[0]), 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--sizes-mb", default=",".join(str(s) for s in SIZES_MB))
    ap.add_argument("--zero-params-mb", type=int, default=512, help="bf16 model size of the ZeroOptimizer case")
    args = ap.parse_args()
    rank, size = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    # every rank is a child of the same launcher process: a file store private to this launch
    store = os.environ.get("GLB_BENCH_STORE", f"/tmp/glb_bench_mixed_precision_{os.getppid()}")
    ctx = gb.init_context(rank, size, path=store, timeout_ms=120000)
    cc = gcu.CudaContext(ctx, local, stage_bytes=64 << 20)
    bf16, f32 = torch.bfloat16, torch.float32
    res = {"world": size, **gpu_info(), "iters": args.iters, "unit": "us per call, max over ranks",
           "l2": "not flushed between passes", "rows": []}
    s = 1.0 / size
    for mb in (int(x) for x in args.sizes_mb.split(",")):
        n = (mb << 20) // 2 // size * size       # bf16 elements of the full parameter vector
        per = n // size
        g16 = cc.empty(n, bf16)
        g16.normal_()
        g32 = cc.empty(n, f32)                   # the upcast temporary of the two-step path
        o32, o16 = torch.empty(per, dtype=f32, device="cuda"), torch.empty(per, dtype=bf16, device="cuda")
        # the bf16 vector that every cast call reads or writes fits L2: repeated passes hit it there
        row = {"bf16_params_mb": mb, "l2_resident": mb < L2_MB}
        # (a) reduce_scatter of bf16 gradients into an fp32 shard
        row["rs_cast_bf16_to_f32"] = timed(lambda: cc.reduce_scatter(o32, g16, scale=s), cc, args.iters, args.warmup)

        def upcast_rs():
            g32.copy_(g16)
            cc.reduce_scatter(o32, g32, scale=s)

        row["rs_upcast_then_f32"] = timed(upcast_rs, cc, args.iters, args.warmup)
        row["rs_bf16"] = timed(lambda: cc.reduce_scatter(o16, g16, scale=s), cc, args.iters, args.warmup)
        # (b) allgather of the fp32 master shard into bf16 parameters
        m32 = torch.randn(per, dtype=f32, device="cuda")
        m16 = torch.empty(per, dtype=bf16, device="cuda")
        row["ag_cast_f32_to_bf16"] = timed(lambda: cc.allgather(g16, m32), cc, args.iters, args.warmup)

        def ag_then_downcast():
            cc.allgather(g32, m32)
            g16.copy_(g32)

        row["ag_f32_then_downcast"] = timed(ag_then_downcast, cc, args.iters, args.warmup)

        def downcast_then_ag():
            m16.copy_(m32)
            cc.allgather(g16, m16)

        row["ag_downcast_then_bf16"] = timed(downcast_then_ag, cc, args.iters, args.warmup)
        res["rows"].append(row)
        del g16, g32, o32, o16, m32, m16
        torch.cuda.empty_cache()
    # (c) ZeroOptimizer.step() on a bf16 model larger than L2
    width = 4096
    layers = max(1, (args.zero_params_mb << 20) // 2 // (width * width))
    for master in (None, f32):
        torch.manual_seed(0)
        model = torch.nn.Sequential(*[torch.nn.Linear(width, width, bias=False) for _ in range(layers)]).to(bf16).cuda()
        zo = ZeroOptimizer(ctx, cc, model.parameters(), torch.optim.AdamW, master_dtype=master, lr=1e-4)
        for p in model.parameters():
            p.grad.normal_()
        key = "zero_step_master_f32" if master is not None else "zero_step_bf16"
        res[key] = timed(zo.step, cc, max(3, args.iters // 4), 2)
        res["zero_model_mb"] = layers * width * width * 2 >> 20
        del zo, model
        torch.cuda.empty_cache()
    cc.synchronize()
    cc.barrier()
    cc.synchronize()
    if rank == 0:
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
