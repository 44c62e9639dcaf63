"""Shared pieces of the mixed-precision reduce_scatter / allgather tests: the CPU model of the
converting allgather, input generators, and the single-process emulation of
``ZeroOptimizer(master_dtype=torch.float32)`` that the threaded and multi-process checks
compare against. Imported by the test modules and the one-process-per-GPU worker."""
from __future__ import annotations

import numpy as np

import reduction_oracle as ro

PAIRS = (("f32", "bf16"), ("f32", "f16"), ("bf16", "f32"), ("f16", "f32"))


def convert_bits(bits: np.ndarray, src, dst) -> np.ndarray:
    """The converting allgather's model: one round-to-nearest-even conversion (exact when
    widening) of raw ``src`` bits to raw ``dst`` bits."""
    with np.errstate(over="ignore", invalid="ignore"):
        return ro.to_bits(ro.from_bits(bits, src), dst)


def random_bits(n: int, d, seed: int) -> np.ndarray:
    """Uniformly random raw bits of dtype ``d``: every class of value (zeros, subnormals, normals
    near both ends of the range, Inf, NaN) shows up, and f32 values far beyond the f16 range."""
    d = ro.dtype(d)
    rng = np.random.default_rng(seed)
    return rng.integers(0, 2**d.width, n, dtype=np.uint64).astype(d.bits)


def tie_bits(n: int, d, seed: int) -> np.ndarray:
    """f32 bits exactly halfway between two neighbouring values of the 16-bit type ``d``."""
    low = 0x8000 if ro.dtype(d) is ro.BF16 else 0x1000
    rng = np.random.default_rng(seed)
    # f16: normal f16 magnitudes only (2**-14 up to below the overflow threshold)
    lo, hi = (0x00800000, 0x7F000000) if low == 0x8000 else (0x38800000, 0x477F0000)
    u = (rng.integers(lo, hi, n, dtype=np.int64) & ~(2 * low - 1)) | low
    sign = rng.integers(0, 2, n, dtype=np.int64) << 31
    return (u | sign).astype(np.uint32)


def edge_values(src) -> np.ndarray:
    """Values of ``src`` that exercise the conversion: signed zeros, infinities, NaN, values that
    overflow or underflow f16, subnormals and the largest finite values."""
    common = [-0.0, 0.0, np.inf, -np.inf, np.nan, 1.0, -2.5]
    if ro.dtype(src) is ro.F32:
        extra = [65504.0, 65519.0, 65520.0, 1e6, -1e6, 3.0e38, 1e-8, 6e-8, 3e-5, 1e-40, 2.0**-126, 1.0 + 2.0**-8,
                 1.0 + 3 * 2.0**-9]
    elif ro.dtype(src) is ro.F16:
        extra = [65504.0, -65504.0, 2.0**-24, 3 * 2.0**-24, 2.0**-14, 1000.0]
    else:
        extra = [3.0e38, -3.0e38, 2.0**-133, 2.0**-126, 1e10]
    v = np.array(common + extra, dtype=np.float64)
    return ro.from_bits(ro.to_bits(v, src), src)  # representable in src


def zero_emulation(grads_per_rank, p0, steps: int, lr: float = 1e-2):
    """What ``ZeroOptimizer(master_dtype=torch.float32)`` over AdamW computes, in one process:
    per-rank bf16 gradients are averaged in fp32 (sum in fp32, times 1/P), an fp32 AdamW steps
    the full fp32 master vector, and the bf16 parameters are its round-to-nearest-even downcast.
    ``grads_per_rank[s][r]``: rank r's bf16 gradient at step s (flat). Returns (master, bf16)."""
    import torch

    P = len(grads_per_rank[0])
    master = torch.nn.Parameter(p0.float().clone())
    opt = torch.optim.AdamW([master], lr=lr)
    for s in range(steps):
        acc = grads_per_rank[s][0].float().clone()
        for r in range(1, P):
            acc += grads_per_rank[s][r].float()
        master.grad = acc * np.float32(1.0 / P)
        opt.step()
    return master.detach().clone(), master.detach().to(torch.bfloat16)
