"""Bit-exact, launch-checked tests for every compiled pointwise-GEMM and depthwise-conv kernel variant.

Exact arithmetic.  Activations, weights and residuals are small integers, scales are powers of two and shifts small
multiples of a power of two, with the sparsity set from the reduction length so that the sum of |products| of every
output is at most 2^20.  Every partial sum is then an integer that fp32 holds exactly, whatever the summation order,
including the truncating largest-term-aligned summation of the tensor cores, and scale/shift, the ReLU6 clamp and the
residual add are exact in fp32 too.  The only rounding left is the final one to the storage type, so the expected
output is known bit for bit: a float64 evaluation on the device, then float64 -> float32 (exact, asserted) -> storage
type (round to nearest even).  Most pre-rounding values are representable in the storage type, so a wrong tap, channel
or time index cannot hide in the output rounding; a share of them is not, which exercises ties and the rounding mode.
Cancellation cases put integers near 2^15 into the first K block (the first taps) and their negation into the last: an
fp32 accumulator keeps the small integers in between exactly, a 16-bit one does not.

Owned outputs.  Every kernel writes into a buffer the test owns, filled with a NaN pattern no kernel produces from
finite data (hardware NaNs are canonical) and framed by guard bands.  An output element a kernel skips stays the
sentinel instead of showing a stale correct value the caching allocator handed back, and a write outside the
allocation changes a guard band.  The pitch padding may be written: the fp32 head (conv_gemm_kernel with OUT_F32)
stores up to the pitch, dw_tc_kernel and dw_simt_kernel store whole 8-step groups, and dw_bulk_kernel and
dw_s2_mma_kernel store a (t, t + 1) pair that starts on the last column.  Inputs carry NaN in their pitch padding.

Launch coverage.  The whole case list runs once more under torch.profiler, and every variant the dispatchers of
conv_gemm.cu and dwconv.cu can select must be among the launched kernels.  Needs a CUDA device (-m gpu).
"""
import math
import re
from dataclasses import dataclass

import pytest
import torch

from voice100_b200 import kernels as K

pytestmark = pytest.mark.gpu
DEV = "cuda"
BF16, F16, F32 = torch.bfloat16, torch.float16, torch.float32
MANT = {BF16: 8, F16: 11}                                 # significand bits of the storage type
SENTINEL = {BF16: 0x7FA5, F16: 0x7D5A, F32: 0x7FA5A5A5}   # non-canonical NaNs
NEG_ZERO = {BF16: -0x8000, F16: -0x8000, F32: -0x80000000}
GUARD_BYTES = 4096
EXACT_LIMIT = 2.0 ** 20          # bound on the sum of |products| of one output (fp32 has a 24-bit significand)
MIN_REPRESENTABLE = 0.70         # share of pre-rounding values the storage type holds exactly, per case


def _bits_type(dtype):
    return torch.int16 if dtype.itemsize == 2 else torch.int32


class Owned:
    """Output buffer of `shape` owned by the test: sentinel-filled, GUARD_BYTES of guard band on both sides."""

    def __init__(self, shape, dtype):
        self.dtype, self.shape = dtype, tuple(shape)
        self.g = GUARD_BYTES // dtype.itemsize
        self.n = math.prod(shape)
        self.raw = torch.full((self.g + self.n + self.g,), SENTINEL[dtype], dtype=_bits_type(dtype), device=DEV)
        self.t = self.raw[self.g:self.g + self.n].view(dtype).view(self.shape)

    def ptr(self):
        return self.t.data_ptr()

    def check(self, valid: torch.Tensor, expect: torch.Tensor, what: str):
        """`valid` = the view of self.t the kernel must write; `expect` = its exact expected value."""
        s = SENTINEL[self.dtype]
        for side, band in (("before", self.raw[:self.g]), ("after", self.raw[self.g + self.n:])):
            n_bad = int((band != s).sum())
            assert n_bad == 0, f"{what}: {n_bad} elements of the guard band {side} the output were written"
        bt = _bits_type(self.dtype)
        got = valid.view(bt)
        n_skip = int((got == s).sum())
        assert n_skip == 0, f"{what}: {n_skip} of {got.numel()} output elements were never written"
        exp = expect.to(self.dtype).view(bt)
        nz = NEG_ZERO[self.dtype]
        got, exp = torch.where(got == nz, 0, got), torch.where(exp == nz, 0, exp)   # -0 == +0
        bad = got != exp
        if bool(bad.any()):
            idx = [int(i) for i in bad.nonzero()[0]]
            g1, e1 = valid[tuple(idx)].item(), expect.to(self.dtype)[tuple(idx)].item()
            raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} outputs differ from the exact result; "
                                 f"first at {idx}: got {g1!r}, expected {e1!r}")


# ------------------------------------------------------------------------------------------------
# exact operands
# ------------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def ints(shape, amp, gen, density=1.0):
    """Integers uniform in [-amp, amp] (float64), each kept with probability `density`."""
    v = torch.randint(-amp, amp + 1, tuple(shape), generator=gen, device=DEV).double()
    if density < 1.0:
        v = v * (torch.rand(tuple(shape), generator=gen, device=DEV, dtype=torch.float64) < density)
    return v


def plan(n_terms, dtype, w_amp=4):
    """(activation amplitude, density) so that a sum of n_terms products x * w (w uniform in [-w_amp, w_amp]) has a
    standard deviation near 2^(m-1), m = the storage type's significand bits."""
    target2 = (0.9 * 2.0 ** (MANT[dtype] - 1)) ** 2
    ew2 = w_amp * (w_amp + 1) / 3.0
    amp = 4
    while amp < 2 ** MANT[dtype] and n_terms * ew2 * amp * (amp + 1) / 3.0 < target2:
        amp *= 2
    return amp, min(1.0, target2 / (n_terms * ew2 * amp * (amp + 1) / 3.0))


def bn_params(C, dtype, relu6, gen, with_scale=True):
    """Per-channel (scale, shift) in float64: scale a power of two, shift a multiple of 1/2.  With ReLU6 the scale maps
    the accumulator's spread onto about [0, 6], fine enough that part of that range needs rounding."""
    if relu6:
        e = -(MANT[dtype] - 2) + torch.randint(0, 2, (C,), generator=gen, device=DEV)
        shift = torch.randint(1, 5, (C,), generator=gen, device=DEV).double()
    else:
        e = torch.randint(-1, 2, (C,), generator=gen, device=DEV)
        shift = torch.randint(-4, 5, (C,), generator=gen, device=DEV).double() / 2
    # (built from Python floats: torch.pow(2.0, e) on the device is not exact for every negative e in float64)
    scale = torch.tensor([2.0 ** int(i) for i in e.tolist()], device=DEV, dtype=torch.float64) if with_scale else None
    return scale, shift


def finish(acc, scale, shift, relu6, res, ch_dim=1):
    """Exact epilogue in float64: scale * acc + shift, clamp to [0, 6], + residual (the kernels' order)."""
    shp = [1] * acc.dim()
    shp[ch_dim] = -1
    v = acc * (scale.view(shp) if scale is not None else 1.0) + shift.view(shp)
    if relu6:
        v = v.clamp(0.0, 6.0)
    return v + res if res is not None else v


def expected(v64, bound, dtype, what):
    """float64 result -> the float32 value the kernel must hold before its final rounding; asserts the exactness
    preconditions and that most values are representable in the storage type."""
    assert float(bound.max()) <= EXACT_LIMIT, f"{what}: operands too large for exact fp32 sums"
    v32 = v64.float()
    assert torch.equal(v32.double(), v64), f"{what}: a value is not exact in float32"
    if dtype in MANT:
        rep = float((v32.to(dtype).float() == v32).double().mean())
        assert rep >= MIN_REPRESENTABLE, f"{what}: only {rep:.2f} of the values are exact in {dtype}"
    return v32


def ncw_in(v64, dtype):
    """float64 integer values [B, C, T] -> pitched 16-bit Ncw whose pitch padding is NaN."""
    B, C, T = v64.shape
    x = K.empty_ncw(B, C, T, v64.device, dtype)
    x.data.fill_(float("nan"))
    x.data[:, :, :T] = v64.to(dtype)
    assert torch.equal(x.data[:, :, :T].double(), v64)
    return x


def store(w64, dtype):
    t = w64.to(dtype).contiguous()
    assert torch.equal(t.double(), w64)
    return t


def _f32(t):
    return None if t is None else t.float().contiguous()


# ------------------------------------------------------------------------------------------------
# cases
# ------------------------------------------------------------------------------------------------
@dataclass
class Case:
    op: str                  # conv1x1 | conv1x1_f32 | conv1d | conv1d_tm | convtranspose | dwconv
    dtype: torch.dtype
    dims: tuple
    relu6: bool = False
    res: bool = False
    scale: bool = True
    cancel: bool = False
    simt: bool = False
    seed: int = 0

    @property
    def id(self):
        flags = [f for f, on in (("relu6", self.relu6), ("res", self.res), ("noscale", not self.scale),
                                 ("cancel", self.cancel), ("simt", self.simt)) if on]
        return "-".join([self.op, "bf16" if self.dtype == BF16 else "fp16", "x".join(map(str, self.dims))] + flags)


def _epi(i):
    """Epilogue variant i (0..7) of conv_gemm.cu: bit 0 ReLU6, bit 1 residual, bit 2 fp16."""
    return dict(relu6=bool(i & 1), res=bool(i & 2), dtype=F16 if i & 4 else BF16)


# (B, C_in, C_out, T): eight shapes per GEMM family, taking epilogue variants 0..7 in turn
GEMM_FAMILIES = {
    # C_out % 256 != 0 and T where 256-column tiles pad no more than 128-column ones
    "plain256": [(2, 72, 200, 129), (3, 264, 24, 255), (1, 8, 2, 256), (2, 2048, 200, 511), (1, 72, 24, 512),
                 (2, 264, 200, 751), (1, 8, 136, 1200), (60, 72, 200, 751)],          # last: 360 tiles > 2 x 148
    "plain128": [(1, 8, 24, 1), (2, 72, 2, 7), (3, 264, 200, 8), (2, 8, 136, 9), (1, 2048, 24, 127),
                 (4, 72, 200, 128), (2, 264, 24, 257), (150, 8, 200, 128)],           # last: 300 tiles
    # C_out % 256 == 0 with C_in that the weights-resident kernel does not take
    "pair256": [(2, 72, 256, 129), (1, 264, 512, 255), (3, 8, 256, 256), (1, 2048, 512, 511), (2, 72, 2048, 512),
                (1, 264, 256, 751), (1, 8, 512, 1200), (80, 72, 512, 256)],           # last: 160 tiles > 148 pairs
    "pair128": [(1, 8, 256, 1), (2, 72, 512, 7), (3, 264, 256, 8), (1, 2048, 256, 9), (2, 72, 2048, 127),
                (1, 264, 512, 128), (2, 8, 256, 257), (1, 72, 512, 1100)],
    # weights resident in tensor memory: C_in <= 512, C_in % 128 == 0, (T / 128) * B units >= 4 per pair
    "wres": [(40, 128, 2048, 129), (18, 256, 2048, 257), (72, 512, 1024, 128), (148, 128, 512, 8),
             (24, 384, 768, 511), (9, 256, 2048, 1100), (36, 128, 2048, 1), (40, 512, 2048, 255)],
}


def _cases():
    cs = []
    for fam, shapes in GEMM_FAMILIES.items():
        for i, dims in enumerate(shapes):
            cs.append(Case("conv1x1", dims=dims, scale=i % 3 != 2, seed=len(cs), **_epi(i)))
    for dims, dtype, res in (((2, 2048, 200, 300), BF16, False), ((2, 2048, 200, 300), F16, True),
                             ((2, 2048, 512, 129), BF16, True), ((2, 2048, 512, 129), F16, False),
                             ((40, 512, 2048, 129), BF16, False), ((40, 512, 2048, 129), F16, True)):
        cs.append(Case("conv1x1", dtype, dims, res=res, cancel=True, seed=len(cs)))
    for dims in ((2, 256, 29, 751), (3, 512, 260, 100), (1, 512, 2, 24), (2, 72, 29, 1)):   # CTC / WORLD heads
        for dtype in (BF16, F16):
            cs.append(Case("conv1x1_f32", dtype, dims, seed=len(cs)))
    # (B, C_in, C_out, T, k, stride, pad): tap stacking + the 1x1 GEMM
    for dims, dtype in (((2, 64, 200, 300, 3, 1, 1), BF16), ((3, 72, 256, 129, 5, 2, 2), F16),
                        ((1, 128, 24, 9, 5, 1, 2), F16), ((2, 8, 2, 5, 3, 2, 0), BF16)):
        cs.append(Case("conv1d", dtype, dims, seed=len(cs)))
    # (C_in, C_out, T, Bp, k): time-major dense conv, N = T * Bp columns
    for dims, dtype in (((64, 256, 40, 8, 3), BF16), ((128, 512, 32, 16, 5), F16), ((64, 200, 96, 8, 1), F16),
                        ((192, 24, 100, 8, 5), BF16)):
        cs.append(Case("conv1d_tm", dtype, dims, seed=len(cs)))
    # (B, C_in, C_out, T): ConvTranspose1d k5 s2
    for dims, dtype in (((2, 64, 200, 129), BF16), ((3, 128, 256, 1), F16), ((1, 64, 24, 300), F16),
                        ((2, 192, 136, 40), BF16)):
        cs.append(Case("convtranspose", dtype, dims, seed=len(cs)))
    # depthwise (B, C, T, k, stride); ReLU6 x dtype in turn inside each group
    dw_groups = [
        # dw_tc_kernel NP = 1 (k <= 33), 2 (k <= 65), 3 (k <= 97): short rows, C % 8 != 0, the N rounding of B
        [(1, 12, 751, 33, 1), (16, 20, 127, 15, 1), (17, 13, 129, 17, 1), (128, 12, 8, 1, 1), (2, 12, 512, 19, 1),
         (2, 16, 511, 19, 1)],
        [(129, 12, 128, 35, 1), (1, 13, 1100, 65, 1), (257, 12, 9, 59, 1), (16, 20, 256, 35, 1)],
        [(17, 12, 751, 67, 1), (1, 13, 257, 97, 1), (128, 12, 7, 97, 1), (129, 12, 1, 67, 1)],
        # dw_bulk_kernel Q = 1 (k = 1), 2 (k <= 17), 3 (k <= 33): T >= 512, C % 8 == 0, odd last chunks
        [(3, 8, 512, 1, 1), (2, 16, 751, 1, 1), (9, 8, 1100, 1, 1), (1, 8, 2100, 1, 1)],
        [(5, 8, 751, 15, 1), (2, 16, 1025, 17, 1), (17, 8, 512, 17, 1), (3, 8, 2049, 15, 1)],
        [(3, 8, 751, 33, 1), (9, 16, 1100, 19, 1), (2, 8, 513, 27, 1), (1, 24, 3001, 33, 1)],
        # dw_s2_mma_kernel: Q 2 / 3 x 7 / 11 prefetched vectors (11 once T_out > 754)
        [(11, 20, 1, 11, 2), (3, 13, 100, 3, 2)], [(2, 20, 1509, 11, 2), (3, 13, 2600, 31, 2)],
        [(5, 20, 1501, 59, 2), (2, 12, 257, 35, 2)], [(2, 20, 3001, 59, 2), (9, 13, 2100, 45, 2)],
        # dw_s2_kernel (stride 2, 61 <= k <= 93) and dw_simt_kernel (stride 1, k >= 99; stride 2, k >= 95)
        [(3, 13, 1501, 61, 2), (2, 20, 257, 93, 2)], [(2, 13, 751, 99, 1), (2, 12, 300, 95, 2)],
    ]
    for group in dw_groups:
        for i, dims in enumerate(group):
            relu6 = bool(i & 2) if len(group) > 2 else i == 0
            cs.append(Case("dwconv", F16 if i & 1 else BF16, dims, relu6=relu6, scale=i != 3, seed=len(cs)))
    for dims, dtype in (((3, 12, 129, 83, 1), F16), ((2, 20, 1501, 11, 2), BF16)):     # forced CUDA-core kernel
        cs.append(Case("dwconv", dtype, dims, relu6=True, simt=True, seed=len(cs)))
    for dims, dtype in (((2, 12, 751, 65, 1), BF16), ((1, 13, 1100, 97, 1), F16),        # dw_tc NP 2 / 3
                        ((2, 13, 1501, 61, 2), F16), ((2, 12, 1501, 99, 1), BF16)):      # dw_s2, dw_simt
        cs.append(Case("dwconv", dtype, dims, cancel=True, seed=len(cs)))
    return cs


CASES = _cases()


# ------------------------------------------------------------------------------------------------
# per-op setup: operands, owned outputs, exact expectation, the direct C call and the wrapper call
# ------------------------------------------------------------------------------------------------
class Prepared:
    def __init__(self, case, with_expect=True):
        self.case = case
        getattr(self, "_" + case.op)(case, _gen(1000 + case.seed), with_expect)

    # ---- pointwise GEMM ----
    def _conv1x1(self, c, gen, with_expect):
        B, C_in, C_out, T = c.dims
        dt = c.dtype
        amp, dens = plan(C_in, dt)
        x = ints((B, C_in, T), amp, gen, dens)
        W = ints((C_out, C_in), 4, gen)
        if c.cancel:
            # integers near 2^15 in channels 0, 1 (first K block), the same values in the last K block against the
            # negated weights: the products cancel only after every K block in between was accumulated
            big = 2.0 ** 15 if dt == BF16 else 2.0 ** 13
            x[:, :64] = 0
            x[:, C_in - 64:] = 0
            x[:, :2] = big * torch.randint(0, 2, (B, 2, T), generator=gen, device=DEV).double().mul_(2).sub_(1)
            x[:, C_in - 64:C_in - 62] = x[:, :2]
            W[:, C_in - 64:C_in - 62] = -W[:, :2]
        scale, shift = bn_params(C_out, dt, c.relu6, gen, c.scale)
        r = ints((B, C_out, T), 8, gen) if c.res else None
        self.x, self.W = ncw_in(x, dt), store(W, dt)
        self.scale, self.shift = _f32(scale), _f32(shift)
        self.r = ncw_in(r, dt) if c.res else None
        self.y = Owned((B, C_out, K.pitch_of(T)), dt)
        if with_expect:
            acc = torch.einsum("oc,bct->bot", W, x)
            bound = torch.einsum("oc,bct->bot", W.abs(), x.abs())
            self.expect = expected(finish(acc, scale, shift, c.relu6, r), bound, dt, c.id)
        self.valid = lambda y: y[:, :, :T]

    def _launch_conv1x1(self, y_ptr):
        c, (B, C_in, C_out, T) = self.case, self.case.dims
        K._call(self.x, "v100_conv1x1", self.x.data.data_ptr(), self.x.pitch, self.W.data_ptr(),
                K._ptr(self.scale), self.shift.data_ptr(), None if self.r is None else self.r.data.data_ptr(), y_ptr,
                K.pitch_of(T), B, C_in, C_out, T, K.ACT_RELU6 if c.relu6 else K.ACT_NONE, K.dt(c.dtype))

    def _wrap_conv1x1(self):
        return K.conv1x1(self.x, self.W, self.scale, self.shift, K.ACT_RELU6 if self.case.relu6 else K.ACT_NONE,
                         self.r).data

    # ---- pointwise GEMM, fp32 head ----
    def _conv1x1_f32(self, c, gen, with_expect):
        B, C_in, C_out, T = c.dims
        amp, dens = plan(C_in, c.dtype)
        x, W = ints((B, C_in, T), amp, gen, dens), ints((C_out, C_in), 4, gen)
        bias = torch.randint(-64, 65, (C_out,), generator=gen, device=DEV).double() / 4
        self.x, self.W, self.bias = ncw_in(x, c.dtype), store(W, c.dtype), _f32(bias)
        self.y = Owned((B, C_out, self.x.pitch), F32)
        if with_expect:
            acc = torch.einsum("oc,bct->bot", W, x)
            bound = torch.einsum("oc,bct->bot", W.abs(), x.abs())
            self.expect = expected(acc + bias[None, :, None], bound, F32, c.id)
        self.valid = lambda y: y[:, :, :T]

    def _launch_conv1x1_f32(self, y_ptr):
        c, (B, C_in, C_out, T) = self.case, self.case.dims
        K._call(self.x, "v100_conv1x1_f32out", self.x.data.data_ptr(), self.x.pitch, self.W.data_ptr(),
                self.bias.data_ptr(), y_ptr, self.x.pitch, B, C_in, C_out, T, K.dt(c.dtype))

    def _wrap_conv1x1_f32(self):
        return K.conv1x1_f32(self.x, self.W, self.bias).data

    # ---- dense Conv1d: tap stacking + GEMM ----
    def _conv1d(self, c, gen, with_expect):
        B, C_in, C_out, T, k, s, pad = c.dims
        T_out = (T + 2 * pad - k) // s + 1
        amp, dens = plan(k * C_in, c.dtype)
        x, Wp = ints((B, C_in, T), amp, gen, dens), ints((C_out, k * C_in), 4, gen)
        bias = torch.randint(-8, 9, (C_out,), generator=gen, device=DEV).double() / 2
        self.x, self.Wp, self.bias = ncw_in(x, c.dtype), store(Wp, c.dtype), _f32(bias)
        self.ws = torch.full((B, k * C_in, K.pitch_of(T_out)), float("nan"), device=DEV, dtype=c.dtype)
        self.y = Owned((B, C_out, K.pitch_of(T_out)), c.dtype)
        if with_expect:
            xp = torch.nn.functional.pad(x, (pad, pad))
            W3 = Wp.view(C_out, k, C_in)
            acc = sum(torch.einsum("oc,bct->bot", W3[:, j], xp[:, :, j:j + s * (T_out - 1) + 1:s]) for j in range(k))
            bound = sum(torch.einsum("oc,bct->bot", W3[:, j].abs(), xp[:, :, j:j + s * (T_out - 1) + 1:s].abs())
                        for j in range(k))
            self.expect = expected(acc + bias[None, :, None], bound, c.dtype, c.id)
        self.valid = lambda y: y[:, :, :T_out]

    def _launch_conv1d(self, y_ptr):
        c, (B, C_in, C_out, T, k, s, pad) = self.case, self.case.dims
        K._call(self.x, "v100_conv1d", self.x.data.data_ptr(), self.x.pitch, self.Wp.data_ptr(), self.bias.data_ptr(),
                self.ws.data_ptr(), y_ptr, self.y.shape[2], B, C_in, C_out, T, k, s, pad, K.dt(c.dtype))

    def _wrap_conv1d(self):
        _, _, _, _, k, s, pad = self.case.dims
        return K.conv1d(self.x, self.Wp, self.bias, k, s, pad).data

    # ---- dense Conv1d on the time-major layout ----
    def _conv1d_tm(self, c, gen, with_expect):
        C_in, C_out, T, Bp, k = c.dims
        amp, dens = plan(k * C_in, c.dtype)
        x, Wp = ints((C_in, T * Bp), amp, gen, dens), ints((C_out, k * C_in), 4, gen)
        bias = torch.randint(-8, 9, (C_out,), generator=gen, device=DEV).double() / 2
        self.x = K.Tm(store(x, c.dtype), Bp, T, Bp)
        self.Wp, self.bias = store(Wp, c.dtype), _f32(bias)
        self.y = Owned((C_out, T * Bp), c.dtype)
        if with_expect:
            p = (k - 1) // 2
            xb = torch.nn.functional.pad(x.view(C_in, T, Bp), (0, 0, p, p))      # [C_in, T + 2p, Bp]
            W3 = Wp.view(C_out, k, C_in)
            acc = sum(torch.einsum("oc,ctb->otb", W3[:, j], xb[:, j:j + T]) for j in range(k))
            bound = sum(torch.einsum("oc,ctb->otb", W3[:, j].abs(), xb[:, j:j + T].abs()) for j in range(k))
            self.expect = expected((acc + bias[:, None, None]).reshape(C_out, T * Bp),
                                   bound, c.dtype, c.id)
        self.valid = lambda y: y

    def _launch_conv1d_tm(self, y_ptr):
        c, (C_in, C_out, T, Bp, k) = self.case, self.case.dims
        K._call(self.x, "v100_conv1d_tm", self.x.data.data_ptr(), self.Wp.data_ptr(), self.bias.data_ptr(), y_ptr,
                C_in, C_out, T, Bp, k, K.dt(c.dtype))

    def _wrap_conv1d_tm(self):
        return K.conv1d_tm(self.x, self.Wp, self.bias, self.case.dims[4]).data

    # ---- ConvTranspose1d k5 s2 ----
    def _convtranspose(self, c, gen, with_expect):
        B, C_in, C_out, T = c.dims
        amp, dens = plan(3 * C_in, c.dtype)
        x, w = ints((B, C_in, T), amp, gen, dens), ints((C_in, C_out, 5), 4, gen)
        bias = torch.randint(-8, 9, (C_out,), generator=gen, device=DEV).double() / 2
        self.x, self.bias = ncw_in(x, c.dtype), _f32(bias)
        self.Wp = store(w.permute(1, 2, 0).reshape(C_out, 5 * C_in), c.dtype)
        self.ws = torch.full((B, 3 * C_in, self.x.pitch), float("nan"), device=DEV, dtype=c.dtype)
        self.y = Owned((B, C_out, K.pitch_of(2 * T - 1)), c.dtype)
        if with_expect:
            # y[o] = b + sum_{k, t: o = 2 t - 2 + k} w[ci, co, k] x[ci, t]   (stride 2, padding 2)
            full = torch.zeros((B, C_out, 2 * T + 4), device=DEV, dtype=torch.float64)
            fabs = torch.zeros_like(full)
            for j in range(5):
                full[:, :, j:j + 2 * T:2] += torch.einsum("io,bit->bot", w[:, :, j], x)
                fabs[:, :, j:j + 2 * T:2] += torch.einsum("io,bit->bot", w[:, :, j].abs(), x.abs())
            acc, bound = full[:, :, 2:2 * T + 1], fabs[:, :, 2:2 * T + 1]
            self.expect = expected(acc + bias[None, :, None], bound, c.dtype, c.id)
        self.valid = lambda y: y[:, :, :2 * T - 1]

    def _launch_convtranspose(self, y_ptr):
        c, (B, C_in, C_out, T) = self.case, self.case.dims
        K._call(self.x, "v100_convtranspose1d_k5s2", self.x.data.data_ptr(), self.x.pitch, self.Wp.data_ptr(),
                self.bias.data_ptr(), self.ws.data_ptr(), y_ptr, self.y.shape[2], B, C_in, C_out, T, K.dt(c.dtype))

    def _wrap_convtranspose(self):
        return K.convtranspose_k5s2(self.x, self.Wp, self.bias).data

    # ---- depthwise ----
    def _dwconv(self, c, gen, with_expect):
        B, C, T, k, s = c.dims
        dt = c.dtype
        T_out = (T - 1) // s + 1
        if c.cancel:
            # taps 0 and k - 1 are +-2^15 (bf16) / 2^13 (fp16) and x has period k - 1: the two products cancel wherever
            # both taps are inside the row, after every tap in between was accumulated
            per = ints((B, C, k - 1), 4, gen)
            x = per.repeat(1, 1, (T + k - 2) // (k - 1))[:, :, :T].contiguous()
            w = ints((C, k), 4, gen)
            big = 2.0 ** 15 if dt == BF16 else 2.0 ** 13
            w[:, 0] = big * torch.randint(0, 2, (C,), generator=gen, device=DEV).double().mul_(2).sub_(1)
            w[:, k - 1] = -w[:, 0]
        else:
            amp, dens = plan(k, dt)
            x, w = ints((B, C, T), amp, gen, dens), ints((C, k), 4, gen)
        scale, shift = bn_params(C, dt, c.relu6, gen, c.scale)
        self.x, self.w, self.scale, self.shift = ncw_in(x, dt), store(w, dt), _f32(scale), _f32(shift)
        self.y = Owned((B, C, K.pitch_of(T_out)), dt)
        if with_expect:
            p = (k - 1) // 2
            xp = torch.nn.functional.pad(x, (p, p))
            acc = torch.zeros((B, C, T_out), device=DEV, dtype=torch.float64)
            bound = torch.zeros_like(acc)
            for j in range(k):
                xs = xp[:, :, j:j + s * (T_out - 1) + 1:s]
                acc += w[None, :, j, None] * xs
                bound += w[None, :, j, None].abs() * xs.abs()
            self.expect = expected(finish(acc, scale, shift, c.relu6, None), bound, dt, c.id)
        self.valid = lambda y: y[:, :, :T_out]

    def _launch_dwconv(self, y_ptr):
        c, (B, C, T, k, s) = self.case, self.case.dims
        K._call(self.x, "v100_dwconv1d_simt" if c.simt else "v100_dwconv1d", self.x.data.data_ptr(), self.x.pitch,
                self.w.data_ptr(), K._ptr(self.scale), self.shift.data_ptr(), y_ptr, self.y.shape[2], B, C, T, k, s,
                K.ACT_RELU6 if c.relu6 else K.ACT_NONE, K.dt(c.dtype))

    def _wrap_dwconv(self):
        c = self.case
        return K.dwconv(self.x, self.w, self.scale, self.shift, c.dims[3], c.dims[4],
                        K.ACT_RELU6 if c.relu6 else K.ACT_NONE, simt=c.simt).data

    # ---- common ----
    def launch(self):
        getattr(self, "_launch_" + self.case.op)(self.y.ptr())

    def run_wrapper(self):
        return getattr(self, "_wrap_" + self.case.op)()

    def check(self):
        self.y.check(self.valid(self.y.t), self.expect, self.case.id)


@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_exact(case):
    p = Prepared(case)
    p.launch()
    torch.cuda.synchronize()
    p.check()


@pytest.mark.parametrize("op", ["conv1x1", "conv1x1_f32", "conv1d", "conv1d_tm", "convtranspose", "dwconv", "simt"])
def test_wrapper_matches_direct_call(op):
    """The Python wrapper of each entry point computes bit for bit what the direct call into owned memory does."""
    case = next(c for c in CASES if (c.op == op and not c.simt or op == "simt" and c.simt) and (c.op != "conv1x1" or c.res))
    p = Prepared(case, with_expect=False)
    p.launch()
    got = p.run_wrapper()
    torch.cuda.synchronize()
    bt = _bits_type(p.y.dtype)
    assert torch.equal(p.valid(got).view(bt), p.valid(p.y.t).view(bt)), case.id


# ------------------------------------------------------------------------------------------------
# launch coverage
# ------------------------------------------------------------------------------------------------
# Every variant the dispatchers select (template arguments as compiled: conv_gemm_kernel<BLOCK_N, N_ACC, OUT_MODE,
# STAGES, EPI>, conv_gemm_pair_kernel<BLOCK_N, STAGES, EPI>, conv_gemm_wres_kernel<STAGES, EPI>, dw_tc_kernel<NP, RELU6,
# DT>, dw_bulk_kernel<Q, RELU6, DT>, dw_s2_mma_kernel<Q, DT, NV>, dw_s2_kernel<DT>, dw_simt_kernel<DT>).  The fp32 head
# has no dtype template argument: both storage types run the same OUT_F32 instantiation.
REQUIRED = sorted(
    [("conv_gemm_kernel", (256, 1, 0, 3, e)) for e in range(8)]
    + [("conv_gemm_kernel", (128, 1, 0, 4, e)) for e in range(8)]
    + [("conv_gemm_pair_kernel", (256, 5, e)) for e in range(8)]
    + [("conv_gemm_pair_kernel", (128, 6, e)) for e in range(8)]
    + [("conv_gemm_wres_kernel", (9, e)) for e in range(8)]
    + [("conv_gemm_kernel", (256, 1, 1, 4, 0)), ("conv_gemm_kernel", (128, 1, 1, 4, 0))]
    + [("conv_gemm_kernel", (128, 2, 0, 4, e)) for e in (0, 4)]
    + [("dw_tc_kernel", (n, r, d)) for n in (1, 2, 3) for r in (0, 1) for d in (0, 1)]
    + [("dw_bulk_kernel", (q, r, d)) for q in (1, 2, 3) for r in (0, 1) for d in (0, 1)]
    + [("dw_s2_mma_kernel", (q, d, nv)) for q in (2, 3) for d in (0, 1) for nv in (7, 11)]
    + [("dw_s2_kernel", (d,)) for d in (0, 1)]
    + [("dw_simt_kernel", (d,)) for d in (0, 1)])


def _template_arg(a):
    a = a.strip()
    if a in ("true", "false"):
        return int(a == "true")
    m = re.fullmatch(r"\(.*\)\s*(-?\d+)|(-?\d+)[a-zA-Z]*", a)      # "(v100::<enum>)0", "0", "0u"
    if m is None:
        raise ValueError(a)
    return int(m.group(1) or m.group(2))


def kernel_variant(name):
    """Demangled kernel name -> (kernel, template arguments) for v100:: kernels, else None."""
    m = re.search(r"v100::(\w+)<([^<>]*)>", name)
    if m is None:
        return None
    try:
        return m.group(1), tuple(_template_arg(a) for a in m.group(2).split(","))
    except ValueError:
        return None


def test_every_compiled_variant_is_launched():
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    prepared = [Prepared(c, with_expect=False) for c in CASES]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for p in prepared:
            p.launch()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if e.device_type == DeviceType.CUDA}
    assert names, ("the profiler recorded no CUDA kernel events at all: launch coverage cannot be checked "
                   "(CUPTI kernel tracing is unavailable)")
    launched = {v for v in map(kernel_variant, names) if v is not None}
    assert launched, f"no v100:: kernel among the {len(names)} recorded kernels: {sorted(names)[:10]}"
    print("\nlaunched variants:\n  " + "\n  ".join(f"{k}<{', '.join(map(str, a))}>" for k, a in sorted(launched)))
    missing = [f"{k}<{', '.join(map(str, a))}>" for k, a in REQUIRED if (k, a) not in launched]
    assert not missing, f"{len(missing)} required kernel variants were never launched: {missing}"
