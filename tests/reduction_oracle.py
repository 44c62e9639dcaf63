"""CPU reference for the CUDA reductions, exact to the bit.

The CUDA data plane promises that 16-bit types accumulate in fp32 and round once, with the
``scale`` epilogue applied to the fp32 accumulator before that rounding (DESIGN.md,
"Numerics"). This module computes what that promise means for a given set of inputs, so a
kernel's output can be compared bit for bit instead of within a tolerance.

The inputs are chosen so that the answer does not depend on the summation order:
``exact_inputs`` draws ``k * 2**e`` with integer ``|k| <= 255`` and ``e`` in ``[-4, 4]``.
Every value is exact in fp16 and bf16, and every partial sum of up to 24 such terms
(8 ranks x 3 local pointers) is a multiple of 2**-4 below 2**17, so it is exact in fp32.
Whatever order a kernel adds in, its fp32 accumulator holds the exact sum; only the final
conversion to a 16-bit type rounds, and it must round to nearest-even exactly once.

Model (``expected``):
  * SUM: exact sum (fp64), to the accumulator type (fp32; fp64 for float64), times
    ``float32(scale)`` in the accumulator type, one round-to-nearest-even cast to the dtype.
  * PRODUCT: same, on data from {+-0.75, +-1, +-1.5, +-2}; products of up to 8 such values are
    exact in fp32 but not in fp16 / bf16.
  * MIN / MAX: exact.
  * Integers: int64 arithmetic, wrapped to the dtype's width (uint8 wraps mod 256).
  * Several local pointers per rank at P > 1: each rank's fold is rounded once to the dtype
    (it is stored in the dtype before the peers read it), then the cross-rank model applies.
    At P = 1 the fused local step is the whole reduction and rounds once.
  * NVLS (``nvls=True``): ``multimem.ld_reduce`` returns the dtype, so a scale is applied to
    the rounded sum and rounded again: ``round(round(sum) * scale)``. For a dyadic scale such
    as 1/P at P = 2, 4, 8 this equals rounding once.
"""
from __future__ import annotations

import itertools
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

SUM, PRODUCT, MAX, MIN = "sum", "product", "max", "min"
OPS = (SUM, PRODUCT, MAX, MIN)


@dataclass(frozen=True)
class Dtype:
    name: str
    bits: type  # unsigned integer type holding the raw bits
    floating: bool
    width: int  # bits

    @property
    def is16(self) -> bool:
        return self.name in ("f16", "bf16")


F16 = Dtype("f16", np.uint16, True, 16)
BF16 = Dtype("bf16", np.uint16, True, 16)
F32 = Dtype("f32", np.uint32, True, 32)
F64 = Dtype("f64", np.uint64, True, 64)
I32 = Dtype("i32", np.uint32, False, 32)
I64 = Dtype("i64", np.uint64, False, 64)
U8 = Dtype("u8", np.uint8, False, 8)
DTYPES = {d.name: d for d in (F16, BF16, F32, F64, I32, I64, U8)}
_INT_NP = {"i32": np.int32, "i64": np.int64, "u8": np.uint8}


def dtype(d) -> Dtype:
    return d if isinstance(d, Dtype) else DTYPES[d]


# ---- conversions --------------------------------------------------------------------------------

def f32_to_bf16_bits(x) -> np.ndarray:
    """Round-to-nearest-even float32 -> bfloat16 (NaN stays NaN)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    u = x.view(np.uint32).astype(np.uint64)
    rounded = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)
    nan = np.isnan(x)
    return np.where(nan, ((u >> 16) | 0x40).astype(np.uint16), rounded)


def bf16_bits_to_f64(b) -> np.ndarray:
    return (np.asarray(b, dtype=np.uint16).astype(np.uint32) << 16).view(np.float32).astype(np.float64)


def to_bits(values, d) -> np.ndarray:
    """Raw bits of ``values`` stored in dtype ``d``. Floating values are rounded once to
    nearest-even from float64 through ``np.float32`` for 16-bit / f32 targets (exact for the
    values this module produces; call ``round_acc`` for the modelled rounding)."""
    d = dtype(d)
    if d is BF16:
        return f32_to_bf16_bits(np.asarray(values, dtype=np.float64).astype(np.float32))
    if d is F16:
        return np.asarray(values, dtype=np.float64).astype(np.float32).astype(np.float16).view(np.uint16)
    if d is F32:
        return np.asarray(values, dtype=np.float64).astype(np.float32).view(np.uint32)
    if d is F64:
        return np.asarray(values, dtype=np.float64).view(np.uint64)
    return wrap_int(values, d).astype(_INT_NP[d.name]).view(d.bits)


def from_bits(bits, d) -> np.ndarray:
    """Values (float64 for floating dtypes, int64 for integers) of raw bits."""
    d = dtype(d)
    b = np.ascontiguousarray(bits, dtype=d.bits)
    if d is BF16:
        return bf16_bits_to_f64(b)
    if d is F16:
        return b.view(np.float16).astype(np.float64)
    if d is F32:
        return b.view(np.float32).astype(np.float64)
    if d is F64:
        return b.view(np.float64).copy()
    return b.view(_INT_NP[d.name]).astype(np.int64)


def round_acc(acc, d) -> np.ndarray:
    """One rounding of an accumulator (float32 for 16-bit and f32 dtypes, float64 for f64) to
    dtype ``d``; returns raw bits."""
    d = dtype(d)
    if d is BF16:
        return f32_to_bf16_bits(np.asarray(acc, dtype=np.float32))
    if d is F16:
        with np.errstate(over="ignore"):  # overflow to Inf is the correct rounding
            return np.asarray(acc, dtype=np.float32).astype(np.float16).view(np.uint16)
    if d is F32:
        return np.ascontiguousarray(acc, dtype=np.float32).view(np.uint32)
    if d is F64:
        return np.ascontiguousarray(acc, dtype=np.float64).view(np.uint64)
    raise TypeError(f"round_acc: {d.name} is not floating")


def wrap_int(v, d) -> np.ndarray:
    """int64 values wrapped to the width and signedness of integer dtype ``d``."""
    d = dtype(d)
    v = np.asarray(v, dtype=np.int64)
    if d is U8:
        return v & 0xFF
    if d is I32:
        return ((v + 2**31) & 0xFFFFFFFF) - 2**31
    return v


def acc_type(d):
    return np.float64 if dtype(d) is F64 else np.float32


# ---- inputs -------------------------------------------------------------------------------------

PRODUCT_VALUES = np.array([-2.0, -1.5, -1.0, -0.75, 0.75, 1.0, 1.5, 2.0])


def exact_inputs(P: int, n: int, d, seed: int, op: str = SUM) -> List[np.ndarray]:
    """P arrays of n values (float64 for floating dtypes, int64 for integers), each exactly
    representable in ``d``, whose reduction by ``op`` is exact in the accumulator type."""
    d = dtype(d)
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(P):
        if d.floating:
            if op == PRODUCT:
                v = PRODUCT_VALUES[rng.integers(0, len(PRODUCT_VALUES), n)]
            else:
                v = rng.integers(-255, 256, n).astype(np.float64) * np.exp2(rng.integers(-4, 5, n))
        elif op == PRODUCT:
            v = rng.choice(np.array([-3, -2, -1, 1, 2, 3], dtype=np.int64), n)
        elif d is U8:
            v = rng.integers(0, 256, n, dtype=np.int64)
        elif d is I32:
            v = rng.integers(-(2**20), 2**20, n, dtype=np.int64)
        else:
            # above 2**53 and odd: a path through double loses the low bits; 24 terms stay
            # below 2**63
            v = rng.integers(-(2**58), 2**58, n, dtype=np.int64) | 1
        out.append(wrap_int(v, d) if d is U8 else v)
    return out


# ---- model --------------------------------------------------------------------------------------

def _fold(vals: Sequence[np.ndarray], op: str) -> np.ndarray:
    """Left fold starting from the first operand (so -0.0 + -0.0 stays -0.0)."""
    acc = np.array(vals[0], copy=True)
    for v in vals[1:]:
        if op == SUM:
            acc = acc + v
        elif op == PRODUCT:
            acc = acc * v
        elif op == MAX:
            acc = np.where(v > acc, v, acc)
        else:
            acc = np.where(v < acc, v, acc)
    return acc


def _reduce_once(vals: Sequence[np.ndarray], op: str, scale: float, d: Dtype, out: Dtype, nvls: bool) -> np.ndarray:
    """One fused reduction of ``vals`` (values of ``d``) rounded to ``out``; raw bits."""
    if not d.floating:
        assert scale == 1.0, "integer buffers take no scale"
        with np.errstate(over="ignore"):
            return to_bits(wrap_int(_fold([np.asarray(v, dtype=np.int64) for v in vals], op), out), out)
    A = acc_type(d)
    with np.errstate(invalid="ignore", over="ignore"):
        exact = _fold([np.asarray(v, dtype=np.float64) for v in vals], op)
        acc = exact.astype(A)
        if nvls and out.is16 and scale != 1.0:
            acc = from_bits(round_acc(acc, out), out).astype(A)
        if scale != 1.0:
            acc = (acc * A(np.float32(scale))).astype(A)
    return round_acc(acc, out)


def expected(inputs: Sequence[np.ndarray], op: str, scale: float, d, *, ptrs: int = 1, out=None,
             nvls: bool = False) -> np.ndarray:
    """Raw bits every rank must hold after the reduction of ``inputs``.

    ``inputs`` is rank-major: ``len(inputs) == P * ptrs``, entry ``r * ptrs + k`` is local
    pointer k of rank r. ``out`` is the output dtype of a cast epilogue (default: ``d``)."""
    d = dtype(d)
    out = d if out is None else dtype(out)
    assert len(inputs) % ptrs == 0
    P = len(inputs) // ptrs
    if ptrs > 1 and P > 1:
        folded = [from_bits(_reduce_once(inputs[r * ptrs:(r + 1) * ptrs], op, 1.0, d, d, False), d) for r in range(P)]
        return _reduce_once(folded, op, scale, d, out, nvls)
    return _reduce_once(inputs, op, scale, d, out, nvls)


def expected_per_add(inputs: Sequence[np.ndarray], op: str, scale: float, d) -> np.ndarray:
    """What a scalar path that rounds to the dtype after every pairwise step and again after
    the scale computes (the defect the bitwise tests exist to catch)."""
    d = dtype(d)
    acc = to_bits(inputs[0], d)
    for v in inputs[1:]:
        acc = _reduce_once([from_bits(acc, d), v], op, 1.0, d, d, False)
    if scale != 1.0:
        acc = _reduce_once([from_bits(acc, d)], op, scale, d, d, False)
    return acc


# ---- comparison ---------------------------------------------------------------------------------

def _ordered(bits: np.ndarray, d: Dtype) -> np.ndarray:
    """Integers whose difference is the distance in ulps (sign-magnitude -> two's complement)."""
    if not d.floating:
        return from_bits(bits, d).astype(object) if d is I64 else from_bits(bits, d)
    b = bits.astype(np.uint64).astype(object) if d is F64 else bits.astype(np.int64)
    sign = 1 << (d.width - 1)
    if d is F64:
        return np.array([-(x & (sign - 1)) if x & sign else x for x in b], dtype=object)
    return np.where(b & sign, -(b & (sign - 1)), b)


def isnan_bits(bits: np.ndarray, d) -> np.ndarray:
    d = dtype(d)
    if not d.floating:
        return np.zeros(bits.shape, dtype=bool)
    return np.isnan(from_bits(bits, d))


def mismatch(got: np.ndarray, want: np.ndarray, d) -> Optional[str]:
    """None when the raw bits agree (any NaN matches any NaN); otherwise a description with
    the mismatch count, the first index and the largest distance in ulps."""
    d = dtype(d)
    got = np.ascontiguousarray(got).view(d.bits).reshape(-1)
    want = np.ascontiguousarray(want).view(d.bits).reshape(-1)
    if got.shape != want.shape:
        return f"shape {got.shape} != {want.shape}"
    bad = got != want
    bad &= ~(isnan_bits(got, d) & isnan_bits(want, d))
    if not bad.any():
        return None
    idx = np.flatnonzero(bad)
    i = int(idx[0])
    dist = np.abs(_ordered(got[idx], d) - _ordered(want[idx], d))
    return (f"{len(idx)} of {len(got)} elements differ; first at {i}: got {from_bits(got[i:i + 1], d)[0]!r} "
            f"(0x{int(got[i]):x}), want {from_bits(want[i:i + 1], d)[0]!r} (0x{int(want[i]):x}); "
            f"largest distance {max(dist)} ulp")


def assert_bitwise(got: np.ndarray, want: np.ndarray, d, what: str = "") -> None:
    msg = mismatch(got, want, d)
    if msg is not None:
        raise AssertionError(f"{what}: {msg}" if what else msg)


def ulp_error(got_bits: np.ndarray, exact: np.ndarray, d) -> np.ndarray:
    """|got - exact| in units of the dtype's spacing in the binade of max(|got|, |exact|)
    (exact given in float64)."""
    d = dtype(d)
    mant = {"f16": 10, "bf16": 7, "f32": 23, "f64": 52}[d.name]
    emin = {"f16": -14, "bf16": -126, "f32": -126, "f64": -1022}[d.name]
    got = from_bits(got_bits, d)
    mag = np.maximum(np.maximum(np.abs(exact), np.abs(got)), np.finfo(np.float64).tiny)
    e = np.maximum(np.floor(np.log2(mag)), emin)
    return np.abs(got - exact) / np.exp2(e - mant)


def permutations_for(P: int, rng: Optional[np.random.Generator] = None, samples: int = 64) -> List[Sequence[int]]:
    """Every order for P <= 4, ``samples`` random orders above."""
    if P <= 4:
        return list(itertools.permutations(range(P)))
    rng = rng or np.random.default_rng(0)
    return [list(rng.permutation(P)) for _ in range(samples)]


def f32_sum_in_order(vals: Sequence[np.ndarray], order: Sequence[int]) -> np.ndarray:
    acc = np.asarray(vals[order[0]], dtype=np.float32)
    for i in order[1:]:
        acc = (acc + np.asarray(vals[i], dtype=np.float32)).astype(np.float32)
    return acc
