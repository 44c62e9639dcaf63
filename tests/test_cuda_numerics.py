"""Bit-exact numerics of every CUDA reduction kernel against ``reduction_oracle``.

The CPU self-tests at the top check the oracle itself (no GPU needed): its inputs are exact,
its fp32 sums do not depend on order, and it tells a kernel that rounds once from one that
rounds to 16 bits after every add. The GPU tests run threads as ranks on cuda:0, one
``spawn_threads`` call per rank count, and compare raw output bits with the oracle. A rank
never raises on a mismatch (its peers would be left waiting inside a collective): it
collects the failures and the main thread reports them all.
"""
import hashlib
import os
import subprocess
import sys
import tempfile
import zlib

import numpy as np
import pytest

import reduction_oracle as ro


# ---- oracle self-tests (CPU) ---------------------------------------------------------------------

@pytest.mark.parametrize("name", ["f16", "bf16", "f32", "f64", "i32", "i64", "u8"])
def test_oracle_inputs_are_representable(name):
    d = ro.dtype(name)
    for op in (ro.SUM, ro.PRODUCT):
        for x in ro.exact_inputs(24, 4096, d, seed=1, op=op):
            back = ro.from_bits(ro.to_bits(x, d), d)
            assert np.array_equal(back, x), name
    if name == "i64":
        x = ro.exact_inputs(1, 4096, d, seed=1)[0]
        assert (np.abs(x) > 2**53).mean() > 0.9
        assert not np.array_equal(x.astype(np.float64).astype(np.int64), x)  # a double round trip loses bits


@pytest.mark.parametrize("P", [2, 3, 4, 8, 24])
def test_oracle_fp32_sums_are_order_independent(P):
    vals = ro.exact_inputs(P, 20000, "f32", seed=P)
    exact = np.sum(np.stack(vals), axis=0, dtype=np.float64)
    assert np.array_equal(exact.astype(np.float32).astype(np.float64), exact)
    for order in ro.permutations_for(P, np.random.default_rng(P), samples=32):
        assert np.array_equal(ro.f32_sum_in_order(vals, order).astype(np.float64), exact), order
    # products of up to 8 factors are exact in fp32 as well
    pv = ro.exact_inputs(min(P, 8), 20000, "f32", seed=P, op=ro.PRODUCT)
    exact_p = np.prod(np.stack(pv), axis=0, dtype=np.float64)
    assert np.array_equal(exact_p.astype(np.float32).astype(np.float64), exact_p)


@pytest.mark.parametrize("name,P,scale", [("bf16", 3, 1.0), ("bf16", 4, 1.0), ("bf16", 8, 1.0), ("f16", 3, 1.0),
                                          ("f16", 4, 1.0), ("f16", 8, 1.0), ("bf16", 2, 0.3), ("f16", 2, 0.3),
                                          ("bf16", 2, 1 / 3), ("f16", 2, 1 / 3)])
def test_oracle_catches_per_add_rounding(name, P, scale):
    """A scalar path that rounds to 16 bits after every add (and again after the scale)
    disagrees with the once-rounded model on these inputs, so the GPU tests would see it."""
    vals = ro.exact_inputs(P, 4096, name, seed=11)
    want = ro.expected(vals, ro.SUM, scale, name)
    got = ro.expected_per_add(vals, ro.SUM, scale, name)
    msg = ro.mismatch(got, want, name)
    assert msg is not None and "largest distance" in msg
    with pytest.raises(AssertionError):
        ro.assert_bitwise(got, want, name)


@pytest.mark.parametrize("name", ["f32", "f64", "i32", "i64", "u8"])
def test_oracle_per_add_is_exact_for_wide_types(name):
    """Where every partial is exact the two models agree: the 16-bit cases above fail for
    the reason they test and nothing else."""
    P = 8
    vals = ro.exact_inputs(P, 4096, name, seed=5)
    ro.assert_bitwise(ro.expected_per_add(vals, ro.SUM, 1.0, name), ro.expected(vals, ro.SUM, 1.0, name), name)


def _ties(rng, low):
    """float32 values whose bits below the 16-bit type's last mantissa bit are exactly half."""
    u = (rng.integers(0x00800000, 0x7F000000, 20000, dtype=np.int64) & ~(2 * low - 1)) | low
    return u.astype(np.uint32).view(np.float32)


def test_oracle_rounding_matches_torch():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(3)
    x = np.concatenate([rng.standard_normal(100000).astype(np.float32),
                        # exact ties for bf16 and f16
                        _ties(rng, 0x8000),  # halfway between two bf16 values
                        _ties(rng, 0x1000),  # halfway between two f16 values
                        np.float32([0.0, -0.0, np.inf, -np.inf, 65519.0, 65520.0, 1e-8, 6e-8, 3e-5])])
    t = torch.from_numpy(x)
    assert np.array_equal(ro.round_acc(x, "bf16"), t.to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16))
    assert np.array_equal(ro.round_acc(x, "f16"), t.to(torch.float16).view(torch.int16).numpy().view(np.uint16))


def test_oracle_edge_values():
    def v(*xs):
        return [np.array([x]) for x in xs]

    for name in ("f16", "bf16", "f32"):
        val = lambda bits: float(ro.from_bits(bits, name)[0])  # noqa: E731
        assert ro.to_bits([-0.0], name)[0] == ro.expected(v(-0.0, -0.0, -0.0), ro.SUM, 1.0, name)[0]
        assert val(ro.expected(v(60000.0, 60000.0, -60000.0, -60000.0), ro.SUM, 1.0, name)) == 0.0
        assert val(ro.expected(v(np.inf, 1.0, 2.0), ro.SUM, 1.0, name)) == np.inf
        assert np.isnan(val(ro.expected(v(np.inf, -np.inf), ro.SUM, 1.0, name)))
        assert np.isnan(val(ro.expected(v(1.0, np.nan, 2.0), ro.SUM, 0.5, name)))
    # fp16 subnormals summing across the subnormal / normal boundary (2**-14)
    sub = [np.array([600 * 2.0**-24]), np.array([700 * 2.0**-24])]
    assert float(ro.from_bits(ro.expected(sub, ro.SUM, 1.0, "f16"), "f16")[0]) == 1300 * 2.0**-24
    assert ro.expected_per_add(v(60000.0, 60000.0, -60000.0, -60000.0), ro.SUM, 1.0, "f16") != 0  # Inf: per-add overflows


def test_oracle_mismatch_report():
    want = ro.to_bits(np.array([1.0, 2.0, 3.0, np.nan]), "bf16")
    got = want.copy()
    assert ro.mismatch(got, want, "bf16") is None
    got[3] = ro.to_bits(np.array([-np.nan]), "bf16")[0]  # any NaN matches any NaN
    assert ro.mismatch(got, want, "bf16") is None
    got[1] += 3
    got[2] -= 1
    msg = ro.mismatch(got, want, "bf16")
    assert msg.startswith("2 of 4 elements differ; first at 1") and "largest distance 3 ulp" in msg
    z = ro.to_bits(np.array([0.0]), "f32")
    assert ro.mismatch(ro.to_bits(np.array([-0.0]), "f32"), z, "f32") is not None  # -0.0 is not +0.0
    assert ro.mismatch(np.array([2**62 + 1], dtype=np.uint64), np.array([2**62], dtype=np.uint64), "i64") is not None


def test_oracle_multi_pointer_and_nvls_models():
    """Two roundings where the kernels store an intermediate in the dtype, one elsewhere."""
    vals = ro.exact_inputs(6, 4096, "bf16", seed=2)
    once = ro.expected(vals, ro.SUM, 1.0, "bf16")
    assert np.array_equal(ro.expected(vals, ro.SUM, 1.0, "bf16", ptrs=6), once)  # P = 1: fused, once
    assert not np.array_equal(ro.expected(vals, ro.SUM, 1.0, "bf16", ptrs=3), once)  # P = 2: fold, then reduce
    four = ro.exact_inputs(4, 4096, "bf16", seed=3)
    # a dyadic scale commutes with rounding; 0.3 does not
    assert np.array_equal(ro.expected(four, ro.SUM, 0.25, "bf16", nvls=True), ro.expected(four, ro.SUM, 0.25, "bf16"))
    assert not np.array_equal(ro.expected(four, ro.SUM, 0.3, "bf16", nvls=True), ro.expected(four, ro.SUM, 0.3, "bf16"))


# ---- GPU helpers -----------------------------------------------------------------------------------

def _torch_dtype(name):
    import torch

    return {"f16": torch.float16, "bf16": torch.bfloat16, "f32": torch.float32, "f64": torch.float64,
            "i32": torch.int32, "i64": torch.int64, "u8": torch.uint8}[name]


_SIGNED = {1: np.uint8, 2: np.int16, 4: np.int32, 8: np.int64}


def _upload(dst, bits):
    """Copy raw bits (numpy) into the CUDA tensor ``dst`` of the same element size."""
    import torch

    src = torch.from_numpy(np.ascontiguousarray(bits).view(_SIGNED[bits.dtype.itemsize]))
    dst.view(src.dtype).copy_(src)


def _download(t, name):
    import torch

    es = t.element_size()
    raw = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[es]
    return t.detach().view(raw).cpu().numpy().view(ro.dtype(name).bits)


BUF_BYTES = 4 << 20
KINDS = ("plain", "plain+1", "registered", "symmetric", "symmetric+1")
VARIANTS = ("ll", "one_shot", "two_shot", "pipelined", "auto")
LARGE_VARIANTS = ("two_shot", "pipelined", "auto")
ALL_DTYPES = ("f16", "bf16", "f32", "f64", "i32", "i64", "u8")


class _Bufs:
    """Per-rank buffers, allocated once per context: a plain, a registered and a symmetric
    byte buffer; ``view`` carves a typed tensor out of one, optionally one element off the
    16-byte alignment."""

    def __init__(self, cc):
        import torch

        self.plain = torch.empty(BUF_BYTES, dtype=torch.uint8, device="cuda")
        self.reg = torch.empty(BUF_BYTES, dtype=torch.uint8, device="cuda")
        cc.register(self.reg)
        self.sym = cc.empty(BUF_BYTES, torch.uint8)

    def view(self, kind, name, n, at=0):
        dt = _torch_dtype(name)
        es = np.dtype(ro.dtype(name).bits).itemsize
        base = {"plain": self.plain, "registered": self.reg, "symmetric": self.sym}[kind.split("+")[0]]
        off = at + (es if kind.endswith("+1") else 0)
        assert off + n * es <= BUF_BYTES
        return base[off:off + n * es].view(dt)


class _Data:
    """Oracle inputs and expectations, memoised per (dtype, op, scale) at the largest count:
    every model is elementwise, so a prefix of the inputs has the prefix of the result."""

    def __init__(self, P, n):
        self.P, self.n = P, n
        self._in, self._out = {}, {}

    def inputs(self, name, op, ptrs=1):
        key = (name, op, ptrs)
        if key not in self._in:
            seed = zlib.crc32(f"{name}/{op}/{ptrs}/{self.P}".encode())
            vals = ro.exact_inputs(self.P * ptrs, self.n, name, seed=seed, op=op)
            self._in[key] = (vals, [ro.to_bits(v, name) for v in vals])
        return self._in[key]

    def expected(self, name, op, scale, ptrs=1, out=None):
        key = (name, op, scale, ptrs, out)
        if key not in self._out:
            self._out[key] = ro.expected(self.inputs(name, op, ptrs)[0], op, scale, name, ptrs=ptrs, out=out)
        return self._out[key]


def _run_ranks(P, fn):
    import gloo_b200 as gb

    res = gb.spawn_threads(P, fn, cuda_device=0, timeout_ms=120000)
    failures = [f"rank {r}: {m}" for r, out in enumerate(res) for m in out["fail"]]
    assert not failures, f"{len(failures)} failures:\n" + "\n".join(failures[:40])
    return res


def _context(ctx):
    from gloo_b200.ops import cuda as gcu

    cc = gcu.CudaContext(ctx, 0, stage_bytes=16 << 20)
    cc.set_timeout(60000)
    return cc


def _gop(op):
    import gloo_b200 as gb

    return {ro.SUM: gb.ReduceOp.SUM, ro.PRODUCT: gb.ReduceOp.PRODUCT, ro.MIN: gb.ReduceOp.MIN,
            ro.MAX: gb.ReduceOp.MAX}[op]


def _allreduce_cases(P, ll_max):
    small = sorted({1, 2, 3, 4, 5, 6, 7, 8, 9, 15, 16, 17, 8 * P - 1, 8 * P + 1, 4103})
    cases = []
    for name in ALL_DTYPES:
        d = ro.dtype(name)
        es = np.dtype(d.bits).itemsize
        scales = (1.0, 1.0 / P, 0.3) if d.floating else (1.0,)
        for variant in VARIANTS:
            for kind in KINDS:
                counts = list(small)
                if variant in LARGE_VARIANTS and name in ("f16", "bf16", "f32"):
                    counts += [65537, 300001]
                ok = lambda n: not (variant == "ll" and not kind.startswith("plain") and n * es > ll_max)  # noqa: E731
                for i, n in enumerate(c for c in counts if ok(c)):
                    cases.append((name, ro.SUM, variant, kind, n, scales[i % len(scales)]))
                if variant in ("two_shot", "ll", "pipelined"):
                    for op in (ro.PRODUCT, ro.MIN, ro.MAX):
                        for n in (7, 8 * P + 1, 4103):
                            if ok(n):
                                cases.append((name, op, variant, kind, n, 1.0))
    return cases


# ---- GPU: allreduce ----------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 2, 3, 4, 8])
def test_allreduce_bitwise(P):
    """Every variant x buffer kind x dtype x op x count against the once-rounded model, then
    randn fp32 / bf16 data: every rank must hold the same bytes."""

    def fn(ctx):
        import torch

        cc = _context(ctx)
        bufs = _Bufs(cc)
        data = _Data(P, 300001)
        fail, ran = [], 0
        for name, op, variant, kind, n, scale in _allreduce_cases(P, cc.pc.ll_max_bytes()):
            t = bufs.view(kind, name, n)
            _upload(t, data.inputs(name, op)[1][ctx.rank][:n])
            cc.allreduce(t, op=_gop(op), algo=variant, scale=scale)
            cc.synchronize()
            msg = ro.mismatch(_download(t, name), data.expected(name, op, scale)[:n], name)
            ran += 1
            if msg:
                fail.append(f"allreduce {name} {op} {variant} {kind} n={n} scale={scale:.4g}: {msg}")
        digests = []
        g = torch.Generator().manual_seed(1000 + ctx.rank)
        for name in ("f32", "bf16"):
            for variant in VARIANTS:
                for kind in ("plain", "registered", "symmetric+1"):
                    for n in (4103, 300001):
                        if variant in ("ll", "one_shot") and n > 4103:
                            continue
                        if variant == "ll" and not kind.startswith("plain") and n * 4 > cc.pc.ll_max_bytes():
                            continue
                        t = bufs.view(kind, name, n)
                        t.copy_(torch.randn(n, generator=g).to(t.dtype))
                        cc.allreduce(t, algo=variant, average=True)
                        cc.synchronize()
                        digests.append(hashlib.sha1(_download(t, name).tobytes()).hexdigest())
        cc.pc.host_barrier()
        return {"fail": fail, "ran": ran, "digests": digests}

    res = _run_ranks(P, fn)
    assert res[0]["ran"] > 1000
    assert all(r["digests"] == res[0]["digests"] for r in res), "ranks disagree on randn data"


# ---- GPU: reduce_scatter / reduce ---------------------------------------------------------------------

def _rs_tables(P):
    """(label, counts per rank): LL-sized equal shares, the default split of an uneven count,
    and a skewed table whose shares start at offsets that are not 16-byte aligned."""
    tables = [("ll", [100] * P), ("even", [20000] * P), ("uneven", None)]
    if P == 4:
        tables.append(("skewed", [1, 4103, 17, 60001]))
    return tables


@pytest.mark.gpu
@pytest.mark.parametrize("P", [2, 3, 4, 8])
def test_reduce_scatter_and_reduce_bitwise(P):
    def fn(ctx):
        import torch

        cc = _context(ctx)
        bufs = _Bufs(cc)
        data = _Data(P, 100003 * 2)
        fail, ran = [], 0
        for name in ("f16", "bf16", "f32", "i32"):
            scales = (1.0, 0.3) if ro.dtype(name).floating else (1.0,)
            for label, counts in _rs_tables(P):
                n = 100003 if counts is None else sum(counts)
                if counts is None:
                    base, rem = divmod(n, P)
                    counts = [base + (1 if r < rem else 0) for r in range(P)]
                off = sum(counts[:ctx.rank])
                for kind in ("plain", "registered"):
                    for scale in scales:
                        src = bufs.view(kind, name, n)
                        _upload(src, data.inputs(name, ro.SUM)[1][ctx.rank][:n])
                        out = torch.empty(counts[ctx.rank], dtype=_torch_dtype(name), device="cuda")
                        cc.reduce_scatter(out, src, counts=counts, scale=scale)
                        cc.synchronize()
                        want = data.expected(name, ro.SUM, scale)[off:off + counts[ctx.rank]]
                        msg = ro.mismatch(_download(out, name), want, name)
                        ran += 1
                        if msg:
                            fail.append(f"reduce_scatter {name} {label} {kind} scale={scale}: {msg}")
            # reduce: registered input + output (pull kernel into the root), and staged
            for kind in ("plain", "registered"):
                for n in (17, 100003):
                    root = P - 1
                    src = bufs.view(kind, name, n)
                    _upload(src, data.inputs(name, ro.SUM)[1][ctx.rank][:n])
                    if kind == "registered":
                        dst = bufs.view(kind, name, n, at=BUF_BYTES // 2)
                    else:
                        dst = torch.empty(n, dtype=_torch_dtype(name), device="cuda")
                    cc.reduce(dst, src, root=root)
                    cc.synchronize()
                    cc.pc.host_barrier()
                    ran += 1
                    if ctx.rank == root:
                        msg = ro.mismatch(_download(dst, name), data.expected(name, ro.SUM, 1.0)[:n], name)
                        if msg:
                            fail.append(f"reduce {name} {kind} n={n}: {msg}")
        cc.pc.host_barrier()
        return {"fail": fail, "ran": ran}

    _run_ranks(P, fn)


# ---- GPU: cast epilogue -----------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("P", [2, 3, 4])
def test_allreduce_cast_bitwise(P):
    """f32 -> bf16 / f16 and back: fp32 accumulation, scale, one rounding to the output type.
    Registered buffers take castAllreduceKernel (its scalar tail when count % 8 != 0 or the
    buffers are 32-byte misaligned); plain tensors take the LL kernel."""
    pairs = [("f32", "bf16"), ("f32", "f16"), ("bf16", "f32"), ("f16", "f32")]

    def fn(ctx):
        import torch

        cc = _context(ctx)
        bufs = _Bufs(cc)
        data = _Data(P, 65537)
        fail, ran = [], 0
        for src_name, dst_name in pairs:
            for kind in ("registered", "registered+1", "plain"):
                for i, n in enumerate((7, 8, 4103, 65537)):
                    scale = (1.0, 1.0 / P, 0.3)[i % 3]
                    if kind == "plain" and n * 4 > cc.pc.ll_max_bytes():
                        continue
                    src = bufs.view(kind, src_name, n)
                    _upload(src, data.inputs(src_name, ro.SUM)[1][ctx.rank][:n])
                    if kind == "plain":
                        dst = torch.empty(n, dtype=_torch_dtype(dst_name), device="cuda")
                    else:
                        dst = bufs.view("symmetric" + kind[len("registered"):], dst_name, n)
                    cc.allreduce(src, out=dst, scale=scale)
                    cc.synchronize()
                    want = data.expected(src_name, ro.SUM, scale, out=dst_name)[:n]
                    msg = ro.mismatch(_download(dst, dst_name), want, dst_name)
                    ran += 1
                    if msg:
                        fail.append(f"cast {src_name}->{dst_name} {kind} n={n} scale={scale:.4g}: {msg}")
        cc.pc.host_barrier()
        return {"fail": fail, "ran": ran}

    _run_ranks(P, fn)


# ---- GPU: multi-pointer classes ------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 2, 4])
def test_multi_pointer_bitwise(P):
    """CudaAllreduceRingChunked with three local pointers: at P = 1 one fused local kernel
    (rounds once), above that the fold is stored in the dtype and then reduced (rounds twice)."""

    def fn(ctx):
        import torch

        from gloo_b200.ops import cuda as gcu

        data = _Data(P, 65537)
        fail, ran = [], 0
        for name in ("f16", "bf16", "f32"):
            for shift in (0, 1):
                for i, n in enumerate((17, 4103, 65537)):
                    scale = (1.0, 0.3, 1.0 / (3 * P))[i]
                    backing = [torch.empty(n + 8, dtype=_torch_dtype(name), device="cuda") for _ in range(3)]
                    ts = [b[shift:shift + n] for b in backing]
                    bits = data.inputs(name, ro.SUM, ptrs=3)[1]
                    for k, t in enumerate(ts):
                        _upload(t, bits[ctx.rank * 3 + k][:n])
                    algo = gcu.CudaAllreduceRingChunked(ctx, ts)
                    algo.set_scale(scale)
                    algo.run()
                    torch.cuda.current_stream().synchronize()
                    want = data.expected(name, ro.SUM, scale, ptrs=3)[:n]
                    for k, t in enumerate(ts):
                        msg = ro.mismatch(_download(t, name), want, name)
                        ran += 1
                        if msg:
                            fail.append(f"multi-pointer {name} shift={shift} n={n} scale={scale:.4g} ptr {k}: {msg}")
                    del algo
        gcu._cu.peer_context_for(ctx, 0).host_barrier()
        return {"fail": fail, "ran": ran}

    _run_ranks(P, fn)


# ---- GPU: edge values -------------------------------------------------------------------------------

def _edge_inputs(P, name, n):
    """Per-rank values: -0.0 everywhere; +-60000 (an fp16 partial overflows, the sum is 0);
    Inf + finite; +Inf + -Inf; a NaN; then fp16 subnormals whose sum crosses 2**-14."""
    rng = np.random.default_rng(7)
    out = []
    for r in range(P):
        v = (rng.integers(1, 1024 // P + 200, n) * 2.0**-24).astype(np.float64)
        v[0] = -0.0
        v[1] = 60000.0 if r < P // 2 or P == 1 else -60000.0
        v[2] = np.inf if r == 0 else 1.0
        v[3] = np.inf if r == 0 else (-np.inf if r == 1 else 0.0)
        v[4] = np.nan if r == P - 1 else 1.0
        out.append(ro.from_bits(ro.to_bits(v, name), name))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("P", [2, 4])
def test_edge_values(P):
    def fn(ctx):
        cc = _context(ctx)
        bufs = _Bufs(cc)
        fail, ran = [], 0
        for name in ("f16", "bf16", "f32"):
            for n in (13, 8 * P + 5, 1029):
                vals = _edge_inputs(P, name, n)
                want = ro.expected(vals, ro.SUM, 1.0, name)
                for variant, kind in (("two_shot", "registered"), ("two_shot", "symmetric+1"), ("ll", "plain"),
                                      ("one_shot", "plain+1"), ("pipelined", "plain"), ("auto", "symmetric")):
                    t = bufs.view(kind, name, n)
                    _upload(t, ro.to_bits(vals[ctx.rank], name))
                    cc.allreduce(t, algo=variant)
                    cc.synchronize()
                    msg = ro.mismatch(_download(t, name), want, name)
                    ran += 1
                    if msg:
                        fail.append(f"edge {name} n={n} {variant} {kind}: {msg}")
        cc.pc.host_barrier()
        return {"fail": fail, "ran": ran}

    _run_ranks(P, fn)


# ---- GPU: literal schedules -------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("P", [2, 3, 4, 8])
def test_literal_schedules_bounded(P):
    """literal=True runs the named schedule step by step and stores every step's partial in
    the dtype, as the reference does, so it rounds more than once by design. Bound: each
    element takes P - 1 additions in whatever tree the schedule builds, and each stored
    partial is one rounding of at most half an ulp. With positive inputs every partial is at
    most the final sum, so each rounding error is at most half an ulp of the result's binade:
    |got - exact| <= (P - 1) / 2 ulp.

    Where one rank computes each element and the others copy it (ring_chunked,
    halving_doubling, bcube) every rank must hold the same bytes. The plain ring does not
    have that property: every rank folds the whole vector in its own order (own, r-1, r-2, ...)
    and rounds each step, as the reference's ring does."""
    from gloo_b200.ops import cuda as gcu

    classes = [gcu.CudaAllreduceRing, gcu.CudaAllreduceRingChunked, gcu.CudaAllreduceHalvingDoubling,
               gcu.CudaAllreduceBcube]

    def fn(ctx):
        import torch

        data = _Data(P, 65537)
        fail, ran, digests = [], 0, {}
        for cls in classes:
            for name in ("f16", "bf16", "f32"):
                vals = [np.abs(v) for v in data.inputs(name, ro.SUM)[0]]
                exact = np.sum(np.stack(vals), axis=0, dtype=np.float64)
                for n in (1, 17, 4103, 65537):
                    t = torch.empty(n, dtype=_torch_dtype(name), device="cuda")
                    _upload(t, ro.to_bits(vals[ctx.rank][:n], name))
                    cls(ctx, t, literal=True).run()
                    torch.cuda.current_stream().synchronize()
                    got = _download(t, name)
                    digests.setdefault(cls.__name__, []).append(hashlib.sha1(got.tobytes()).hexdigest())
                    err = ro.ulp_error(got, exact[:n], name)
                    ran += 1
                    if err.max() > (P - 1) / 2:
                        fail.append(f"literal {cls.__name__} {name} n={n}: {err.max()} ulp > {(P - 1) / 2}")
        gcu._cu.peer_context_for(ctx, 0).host_barrier()
        return {"fail": fail, "ran": ran, "digests": digests}

    res = _run_ranks(P, fn)
    for name in ("CudaAllreduceRingChunked", "CudaAllreduceHalvingDoubling", "CudaAllreduceBcube"):
        assert all(r["digests"][name] == res[0]["digests"][name] for r in res), f"ranks disagree after literal {name}"


# ---- multi-GPU: NVLS, hybrid, pipelined over multicast --------------------------------------------------

WORKER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cuda_numerics_worker.py")


def _gpu_count():
    try:
        import torch

        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.multigpu
@pytest.mark.skipif(_gpu_count() < 2, reason="needs >= 2 GPUs")
def test_numerics_one_process_per_gpu():
    n = _gpu_count()
    size = 8 if n >= 8 else (4 if n >= 4 else 2)
    d = tempfile.mkdtemp(prefix="glb_numerics_mp_")
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
