"""Stride-1 depthwise conv on tcgen05 (dw_tc_kernel: the filter's Toeplitz matrix in tensor memory, the utterances of
a batch block as the MMA's N axis, data by zero-filled TMA boxes) against fp32 PyTorch on the same operands and against
the CUDA-core kernel.  Runs only on the GPU box (-m gpu)."""
import math

import pytest
import torch
import torch.nn.functional as F

from voice100_b200 import kernels as K

pytestmark = pytest.mark.gpu
DEV = "cuda"
OUT_TOL = {torch.bfloat16: 1.2e-2, torch.float16: 1.5e-3}   # relative to max|ref|: the output rounding


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def ncw_nan_padded(x, dtype):
    """fp32 [B,C,T] -> pitched 16-bit Ncw whose pitch padding is NaN: it is never data and must not leak."""
    B, C, T = x.shape
    out = K.empty_ncw(B, C, T, x.device, dtype)
    out.data.fill_(float("nan"))
    out.data[:, :, :T] = x.to(dtype)
    return out


def rel_err(got, ref):
    got, ref = got.double(), ref.double()
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def reference(xn, w, scale, shift, k, relu6):
    ref = F.conv1d(xn.valid().float(), w.float()[:, None, :], padding=(k - 1) // 2, groups=w.shape[0])
    ref = ref * (scale[None, :, None] if scale is not None else 1.0) + shift[None, :, None]
    return ref.clamp(0, 6) if relu6 else ref


# (B, C, T, k).  Rows of 512 steps or more with k <= 33 and C % 8 == 0 take dw_bulk_kernel, so those here use C = 12 or
# 20.  B: the N rounding (1 -> 16, 17 -> 32) and partial second / third batch blocks (130, 257); T: shorter than a box, one step around the 128-step tile, the benchmark's 751, a 60 s clip; k: 1 ... 97 across the
# three Toeplitz widths (K_w = 160 for k <= 33, 192 for k <= 65, 224 for k <= 97); C > 148: several channels per CTA,
# both Toeplitz buffers rebuilt.
SHAPES = [(1, 12, 751, 83), (17, 12, 129, 97), (130, 12, 128, 1), (257, 12, 127, 33), (17, 12, 5, 35),
          (1, 12, 1, 65), (3, 12, 3001, 67), (130, 20, 751, 3), (257, 12, 751, 19), (2, 300, 751, 51),
          (5, 12, 1, 97), (40, 12, 200, 85), (3, 8, 1027, 75), (16, 8, 640, 59), (33, 12, 300, 9)]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_dwconv_tc_edges(dtype):
    for B, C, T, k in SHAPES:
        x = rnd(B, C, T, seed=T + k)
        w = rnd(C, k, seed=k, scale=1.0 / math.sqrt(k)).to(dtype)
        scale, shift = torch.rand(C, device=DEV) + 0.5, torch.randn(C, device=DEV) * 0.2
        xn = ncw_nan_padded(x, dtype)
        y = K.dwconv(xn, w, scale, shift, k, 1, K.ACT_RELU6)
        got = y.valid().float()
        assert torch.isfinite(got).all(), (B, C, T, k)
        assert rel_err(got, reference(xn, w, scale, shift, k, True)) < OUT_TOL[dtype], (B, C, T, k)
        y = K.dwconv(xn, w, None, shift, k, 1, K.ACT_NONE)                     # no scale, no activation
        assert rel_err(y.valid().float(), reference(xn, w, None, shift, k, False)) < OUT_TOL[dtype], (B, C, T, k)


def test_dwconv_tc_model_shape_matches_simt():
    """The longest filter of asr_en_base at the benchmark's shape, against the CUDA-core kernel and fp32 PyTorch."""
    B, C, T, k = 256, 2048, 751, 83
    x = rnd(B, C, T, seed=83).abs()
    w = rnd(C, k, seed=84, scale=1.0 / math.sqrt(k)).to(torch.bfloat16)
    scale, shift = torch.rand(C, device=DEV) + 0.5, torch.randn(C, device=DEV) * 0.2
    xn = ncw_nan_padded(x, torch.bfloat16)
    got = K.dwconv(xn, w, scale, shift, k, 1, K.ACT_RELU6).valid().float()
    simt = K.dwconv(xn, w, scale, shift, k, 1, K.ACT_RELU6, simt=True).valid().float()
    ref = reference(xn, w, scale, shift, k, True)
    assert torch.isfinite(got).all()
    assert rel_err(got, ref) < OUT_TOL[torch.bfloat16]
    # both round the same fp32 value up to summation order: at most one bf16 step apart
    assert rel_err(got, simt) < OUT_TOL[torch.bfloat16]


def test_dwconv_tc_repeats_are_bit_identical():
    """300 launches must give the first result bit for bit: the mbarrier ring, both accumulators, both Toeplitz buffers
    (C > 148 channels) and both output staging buffers are recycled many times per launch."""
    B, C, T, k = 130, 300, 751, 59
    xn = ncw_nan_padded(rnd(B, C, T, seed=5), torch.bfloat16)
    w = rnd(C, k, seed=6, scale=0.2).to(torch.bfloat16)
    shift = torch.zeros(C, device=DEV)
    first = K.dwconv(xn, w, None, shift, k, 1, K.ACT_NONE)
    assert rel_err(first.valid().float(), reference(xn, w, None, shift, k, False)) < OUT_TOL[torch.bfloat16]
    n_bad = torch.zeros((), device=DEV, dtype=torch.int64)
    for _ in range(300):
        n_bad += (K.dwconv(xn, w, None, shift, k, 1, K.ACT_NONE).valid() != first.valid()).sum()
    assert int(n_bad) == 0
