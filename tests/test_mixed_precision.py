"""CPU checks of the mixed-precision sharded-training path: the oracle model of the converting
allgather against torch's ``.to()``, the argument checks of ``CudaContext`` that run before
anything is launched, and ``ZeroOptimizer(master_dtype=torch.float32)`` over threads on a bf16
model against a single-process emulation."""
import numpy as np
import pytest
import torch

import gloo_b200 as gb
import mixed_precision_common as mp
import reduction_oracle as ro

TORCH = {"f16": torch.float16, "bf16": torch.bfloat16, "f32": torch.float32}
RAW = {2: torch.int16, 4: torch.int32}
SIGNED = {2: np.int16, 4: np.int32}


def _torch_convert(bits, src, dst):
    t = torch.from_numpy(np.ascontiguousarray(bits).view(SIGNED[bits.dtype.itemsize])).view(TORCH[src])
    out = t.to(TORCH[dst])
    return out.view(RAW[out.element_size()]).numpy().view(ro.dtype(dst).bits)


@pytest.mark.parametrize("src,dst", mp.PAIRS)
def test_cast_model_matches_torch(src, dst):
    """``ro.to_bits(ro.from_bits(bits, src), dst)`` is what the converting allgather must store; it
    agrees with torch's conversion on random bits (subnormals, Inf, NaN, f16 overflow included),
    on exact ties and on the edge values."""
    parts = [mp.random_bits(200000, src, seed=1), ro.to_bits(mp.edge_values(src), src)]
    if src == "f32":
        parts.append(mp.tie_bits(20000, dst, seed=2))
    bits = np.concatenate(parts)
    want = _torch_convert(bits, src, dst)
    got = mp.convert_bits(bits, src, dst)
    ro.assert_bitwise(got, want, dst, f"{src}->{dst}")
    # NaN must stay NaN (the comparison above accepts any NaN for any NaN)
    assert np.array_equal(ro.isnan_bits(got, dst), ro.isnan_bits(bits, src))
    if src == "f32":
        ties = mp.tie_bits(1000, dst, seed=3)
        # a tie rounds to the even neighbour: the result's last mantissa bit is 0 unless the tie
        # rounded up into the next binade's first value, whose last bit is also 0
        assert not np.any(mp.convert_bits(ties, src, dst) & 1)


def test_cast_model_edge_values():
    f = lambda v, s, d: ro.from_bits(mp.convert_bits(ro.to_bits(np.array([v]), s), s, d), d)[0]  # noqa: E731
    assert f(65520.0, "f32", "f16") == np.inf and f(65519.0, "f32", "f16") == 65504.0
    assert f(-65520.0, "f32", "f16") == -np.inf
    assert f(1e-8, "f32", "f16") == 0.0 and f(6e-8, "f32", "f16") == 2.0**-24
    assert np.signbit(f(-0.0, "f32", "bf16")) and np.signbit(f(-0.0, "bf16", "f32"))
    assert f(3.0e38, "f32", "bf16") == np.inf or abs(f(3.0e38, "f32", "bf16") - 3.0e38) < 1e36
    assert f(2.0**-24, "f16", "f32") == 2.0**-24  # subnormal widens exactly
    assert np.isnan(f(np.nan, "f32", "f16")) and np.isnan(f(np.nan, "bf16", "f32"))


def test_checks_refuse_bad_arguments_without_a_launch():
    """Length and dtype checks of reduce_scatter / allgather(v) raise before the native call."""
    from gloo_b200.ops import cuda as gcu

    class _FakeCC(gcu.CudaContext):
        def __init__(self):  # no PeerContext: any native call would fail with AttributeError
            self.rank, self.size, self._reg = 1, 2, {}

    cc = _FakeCC()
    f32, bf16 = torch.zeros(16), torch.zeros(16, dtype=torch.bfloat16)
    with pytest.raises(ValueError):
        cc.reduce_scatter(torch.zeros(7), torch.zeros(16))                      # output shorter than its share
    with pytest.raises(ValueError):
        cc.reduce_scatter(torch.zeros(7, dtype=torch.bfloat16), f32)            # the overflow of the issue
    with pytest.raises(ValueError):
        cc.reduce_scatter(torch.zeros(8), bf16[:10], counts=[8, 8])             # input shorter than the counts
    with pytest.raises(ValueError):
        cc.reduce_scatter(torch.zeros(8), f32, counts=[8, 8, 0])                # one count per rank
    with pytest.raises(ValueError):
        cc.allgather(torch.zeros(31, dtype=torch.bfloat16), f32)                # output shorter than sum(counts)
    with pytest.raises(ValueError):
        cc.allgatherv(torch.zeros(32), f32[:3], [4, 4])                         # input shorter than my count
    for out, inp in ((torch.zeros(8, dtype=torch.bfloat16), torch.zeros(16, dtype=torch.float16)),
                     (torch.zeros(8, dtype=torch.float64), f32), (torch.zeros(8), torch.zeros(16, dtype=torch.int32))):
        with pytest.raises(TypeError, match="FLOAT32 -> FLOAT16 / BFLOAT16"):
            cc.reduce_scatter(out, inp)
        with pytest.raises(TypeError):
            cc.allgather(torch.zeros(2 * 16, dtype=out.dtype), torch.zeros(16, dtype=inp.dtype))


@pytest.mark.parametrize("dtype", ["float8_e4m3fn", "float8_e5m2", "uint16", "uint32", "complex64"])
def test_same_dtype_allgather_moves_any_dtype(dtype, monkeypatch):
    """A same-dtype allgather(v) of a dtype without a DataType (float8 FSDP parameters, complex,
    unsigned 16/32-bit) reaches the native byte-moving call, as it did before the cast path."""
    from gloo_b200.ops import cuda as gcu

    dt = getattr(torch, dtype, None)
    if dt is None:
        pytest.skip(f"torch has no {dtype}")
    calls = []

    class _Native:
        def allgatherv(self, pc, iptr, optr, sizes, stream):
            calls.append(("allgatherv", sizes))

    class _FakeCC(gcu.CudaContext):
        def __init__(self):
            self.pc, self.rank, self.size, self._reg = None, 0, 2, {}

    monkeypatch.setattr(gcu, "_cu", _Native())
    cc = _FakeCC()
    inp, out = torch.zeros(8, dtype=dt), torch.zeros(16, dtype=dt)
    cc.allgather(out, inp, stream=0)
    cc.allgatherv(out, inp, [8, 8], stream=0)
    es = inp.element_size()
    assert calls == [("allgatherv", [8 * es, 8 * es])] * 2
    with pytest.raises(TypeError):
        cc.allgather(torch.zeros(16, dtype=torch.float32), inp, stream=0)  # no conversion from this dtype


def _model(seed):
    g = torch.Generator().manual_seed(seed)
    m = torch.nn.Sequential(torch.nn.Linear(13, 29), torch.nn.Linear(29, 5))
    with torch.no_grad():
        for p in m.parameters():
            p.copy_(torch.randn(p.shape, generator=g))
    return m.to(torch.bfloat16)


def _flat_grads(m, rank, step):
    g = torch.Generator().manual_seed(1000 * step + rank)
    return [torch.randn(p.shape, generator=g).to(torch.bfloat16) for p in m.parameters()]


@pytest.mark.parametrize("size", [2, 3])
def test_zero_optimizer_master_fp32_matches_emulation(size):
    """bf16 model, fp32 master shard: per-rank bf16 gradients, fp32 average, fp32 AdamW; the bf16
    parameters are within one bf16 ulp of the emulation's downcast."""
    from gloo_b200.parallel import ZeroOptimizer

    steps = 3

    def fn(ctx):
        m = _model(0)
        zo = ZeroOptimizer(ctx, None, m.parameters(), torch.optim.AdamW, master_dtype=torch.float32, lr=1e-2)
        assert zo.shard.dtype == torch.float32 and zo.shard.grad.dtype == torch.float32
        assert zo.flat_param.dtype == torch.bfloat16 and zo.flat_grad.dtype == torch.bfloat16
        for s in range(steps):
            for p, g in zip(m.parameters(), _flat_grads(m, ctx.rank, s)):
                p.grad.copy_(g)
            zo.step()
            zo.zero_grad()
        return zo.shard.detach().clone(), zo.start, [p.detach().clone() for p in m.parameters()], zo._offs, \
            zo.flat_param.numel()

    res = gb.spawn_threads(size, fn)
    m0 = _model(0)
    _, _, _, offs, n = res[0]
    p0 = torch.zeros(n, dtype=torch.bfloat16)
    for p, off in zip(m0.parameters(), offs):
        p0[off:off + p.numel()] = p.detach().reshape(-1)
    grads = []
    for s in range(steps):
        per_rank = []
        for r in range(size):
            flat = torch.zeros(n, dtype=torch.bfloat16)
            for g, off in zip(_flat_grads(m0, r, s), offs):
                flat[off:off + g.numel()] = g.reshape(-1)
            per_rank.append(flat)
        grads.append(per_rank)
    master, bf16 = mp.zero_emulation(grads, p0, steps)
    for shard, start, params, _, _ in res:
        torch.testing.assert_close(shard, master[start:start + shard.numel()], rtol=1e-6, atol=1e-7)
        for p, off in zip(params, offs):
            want = bf16[off:off + p.numel()].view(p.shape)
            ulps = (p.view(torch.int16).int() - want.view(torch.int16).int()).abs()
            assert int(ulps.max()) <= 1, f"bf16 parameters differ by {int(ulps.max())} ulp"
