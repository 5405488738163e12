"""Per-kernel parity on the device: every C-ABI entry point against a plain fp32 PyTorch evaluation of
the same op on the same (bf16-rounded) operands.  Runs only on the GPU box (-m gpu)."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import v100_oracle as orc
from voice100_b200 import kernels as K
from voice100_b200 import synth
from voice100_b200.data_modules import MelSpectrogramAudioTransform

pytestmark = pytest.mark.gpu
DEV = "cuda"


def ncw(x_f32: torch.Tensor, dtype=torch.bfloat16) -> K.Ncw:
    """fp32 [B,C,T] on device -> pitched 16-bit Ncw with NaN poison in the pitch padding."""
    B, C, T = x_f32.shape
    out = K.empty_ncw(B, C, T, x_f32.device, dtype)
    out.data.fill_(float("nan"))
    out.data[:, :, :T] = x_f32.to(dtype)
    return out


DTYPES = [torch.bfloat16, torch.float16]
OUT_TOL = {torch.bfloat16: 1.2e-2, torch.float16: 1.5e-3}   # relative to max|ref|: the output rounding


def rel_err(got, ref):
    got, ref = got.double(), ref.double()
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


# ------------------------------------------------------------------------------------------------
# pointwise GEMM (tcgen05 + TMA)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,C_in,C_out,T,act,res", [
    (1, 64, 128, 64, 0, False),        # one tile, one k-block
    (1, 128, 128, 256, 0, False),      # two k-blocks, full 256 tile
    (2, 64, 256, 1501, 1, False),      # asr layer-0 expand shape (ragged T, ReLU6)
    (3, 256, 1024, 751, 1, False),     # expand
    (3, 1024, 256, 751, 0, True),      # project + residual
    (2, 512, 2048, 300, 1, False),
    (2, 2048, 512, 300, 0, True),
    (5, 256, 256, 100, 0, True),       # BLOCK_N=128 path
    (2, 72, 200, 333, 1, False),       # K not a multiple of 64, C_out not a multiple of 128
    (40, 128, 384, 520, 0, True),      # > 148 tiles: persistent loop + both TMEM buffers reused
    (4, 2048, 512, 751, 0, True),      # pair kernel at the project shape, K = 2048
    (40, 256, 1024, 751, 1, False),    # weights resident in tensor memory (WRES): K = 256, 4 channel blocks
    (48, 512, 2048, 300, 1, False),    # WRES: K = 512 (all 512 TMEM columns), 8 channel blocks
    (128, 128, 512, 300, 0, True),     # WRES: one ring stage per tile, residual
    (64, 384, 768, 130, 1, True),      # WRES: K = 384, 3 channel blocks, ReLU6 + residual
])
@pytest.mark.parametrize("dtype", DTYPES)
def test_conv1x1_matches_torch(B, C_in, C_out, T, act, res, dtype):
    x = rnd(B, C_in, T, seed=1)
    W = rnd(C_out, C_in, seed=2, scale=1.0 / math.sqrt(C_in)).to(dtype)
    scale = (torch.rand(C_out, device=DEV) + 0.5)
    shift = torch.randn(C_out, device=DEV) * 0.3
    r = rnd(B, C_out, T, seed=3) if res else None
    xn, rn = ncw(x, dtype), (ncw(r, dtype) if res else None)
    y = K.conv1x1(xn, W, scale, shift, act, rn)
    torch.cuda.synchronize()
    ref = torch.einsum("oc,bct->bot", W.float(), xn.valid().float()) * scale[None, :, None] + shift[None, :, None]
    if act:
        ref = ref.clamp(0, 6)
    if res:
        ref = ref + rn.valid().float()
    got = y.valid().float()
    assert torch.isfinite(got).all()
    assert rel_err(got, ref) < OUT_TOL[dtype], rel_err(got, ref)   # output rounding: 2^-8 (bf16) / 2^-11 (fp16)


def test_conv_gemm_stress_is_deterministic():
    """compute-sanitizer's racecheck/synccheck cannot vouch for the tcgen05 GEMM (false positives on mbarrier/TMEM
    traffic, profiles/r01_sanitizer.md), so its synchronisation is stressed instead: 1,000 back-to-back launches per
    shape at odd sizes (ragged T, K not a multiple of 64, C_out not a multiple of 128, residual, CTA pairs, more tiles
    than SMs so both TMEM buffers and every smem stage are recycled), alternating with a different-shaped launch on the
    same stream; every result must be bit-identical to the first, which itself matches fp32 PyTorch."""
    shapes = [(2, 72, 200, 333, 1, False), (3, 1024, 256, 751, 0, True), (40, 128, 384, 520, 0, True),
              (2, 512, 2048, 300, 1, False), (7, 264, 136, 77, 1, True), (48, 512, 2048, 300, 1, False),
              (64, 384, 768, 130, 1, True)]
    other_x = ncw(rnd(1, 64, 97, seed=33))
    other_w = rnd(128, 64, seed=34, scale=0.1).to(torch.bfloat16)
    other_b = torch.zeros(128, device=DEV)
    for B, C_in, C_out, T, act, res in shapes:
        x = rnd(B, C_in, T, seed=31)
        W = rnd(C_out, C_in, seed=32, scale=1.0 / math.sqrt(C_in)).to(torch.bfloat16)
        scale, shift = torch.rand(C_out, device=DEV) + 0.5, rnd(C_out, seed=35)
        xn = ncw(x)
        rn = ncw(rnd(B, C_out, T, seed=36)) if res else None
        first = K.conv1x1(xn, W, scale, shift, act, rn)
        ref = F.conv1d(xn.valid().float(), W.float()[:, :, None]) * scale[None, :, None] + shift[None, :, None]
        if act == K.ACT_RELU6:
            ref = ref.clamp(0, 6)
        if res:
            ref = ref + rn.valid().float()
        assert rel_err(first.valid().float(), ref) < OUT_TOL[torch.bfloat16]
        n_bad = torch.zeros((), device=DEV, dtype=torch.int64)
        for it in range(1000):
            y = K.conv1x1(xn, W, scale, shift, act, rn)
            if it % 3 == 0:
                K.conv1x1(other_x, other_w, None, other_b, 0)
            n_bad += (y.valid() != first.valid()).sum()
        assert int(n_bad) == 0, (B, C_in, C_out, T, int(n_bad))


@pytest.mark.parametrize("B,C_in,C_out,T", [(2, 256, 29, 751), (3, 512, 44, 100), (2, 256, 260, 277), (1, 512, 2, 24)])
@pytest.mark.parametrize("dtype", DTYPES)
def test_conv1x1_f32out_matches_torch(B, C_in, C_out, T, dtype):
    x = rnd(B, C_in, T, seed=4)
    W = rnd(C_out, C_in, seed=5, scale=1.0 / math.sqrt(C_in)).to(dtype)
    bias = torch.randn(C_out, device=DEV)
    xn = ncw(x, dtype)
    y = K.conv1x1_f32(xn, W, bias)
    torch.cuda.synchronize()
    ref = torch.einsum("oc,bct->bot", W.float(), xn.valid().float()) + bias[None, :, None]
    assert rel_err(y.valid(), ref) < 1e-4


@pytest.mark.parametrize("B,C_in,C_out,T", [(2, 512, 256, 277), (1, 64, 128, 40), (3, 128, 64, 130)])
@pytest.mark.parametrize("dtype", DTYPES)
def test_convtranspose_matches_torch(B, C_in, C_out, T, dtype):
    x = rnd(B, C_in, T, seed=6)
    w = rnd(C_in, C_out, 5, seed=7, scale=1.0 / math.sqrt(C_in * 2.5)).to(dtype)
    bias = torch.randn(C_out, device=DEV)
    xn = ncw(x, dtype)
    wp = w.permute(1, 2, 0).reshape(C_out, 5 * C_in).contiguous()
    y = K.convtranspose_k5s2(xn, wp, bias)
    torch.cuda.synchronize()
    ref = F.conv_transpose1d(xn.valid().float(), w.float(), bias, stride=2, padding=2)
    assert y.T == 2 * T - 1 == ref.shape[2]
    assert rel_err(y.valid().float(), ref) < OUT_TOL[dtype]


# ------------------------------------------------------------------------------------------------
# depthwise conv (dw_tc_kernel, dw_bulk_kernel, the stride-2 kernels and the CUDA-core dw_simt_kernel)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [5, 7, 11, 17, 19, 27, 29, 33, 35, 51, 59, 65, 67, 75, 83])
@pytest.mark.parametrize("T", [751, 96])
@pytest.mark.parametrize("dtype", DTYPES)
def test_dwconv_mma_matches_torch(k, T, dtype):
    """Stride 1 through the default dispatch -- at T = 751 dw_bulk_kernel for k <= 33 and dw_tc_kernel from k = 35 up, at
    T = 96 dw_tc_kernel for every k -- and through the CUDA-core dw_simt_kernel."""
    B, C = 2, 64
    x = rnd(B, C, T, seed=k).abs()
    w = rnd(C, k, seed=k + 1, scale=1.0 / math.sqrt(k)).to(dtype)
    scale, shift = torch.rand(C, device=DEV) + 0.5, torch.randn(C, device=DEV) * 0.2
    xn = ncw(x, dtype)
    ref = F.conv1d(xn.valid().float(), w.float()[:, None, :], padding=(k - 1) // 2, groups=C)
    ref = (ref * scale[None, :, None] + shift[None, :, None]).clamp(0, 6)
    for simt in (False, True):
        y = K.dwconv(xn, w, scale, shift, k, 1, K.ACT_RELU6, simt=simt)
        torch.cuda.synchronize()
        assert y.T == T
        assert rel_err(y.valid().float(), ref) < OUT_TOL[dtype], ("simt" if simt else "default", rel_err(y.valid().float(), ref))


@pytest.mark.parametrize("dtype", DTYPES)
def test_dwconv_bulk_staging_edges(dtype):
    """Row staging edges of the stride-1 kernels.  dw_bulk_kernel (k <= 33 on rows of 512 steps or more, C % 8 == 0) stages
    each row by ONE cp.async.bulk + mbarrier; it takes (9, 24, 3001, 27), (17, 8, 1029, 11) and (5, 8, 756, 19): clip-length
    residues mod 8 (the bulk copy moves whole 16-byte groups, the last T & 7 samples come by plain loads one row ahead),
    rows of several 1024-output chunks with a partial last one, batches that are not a multiple of the 8 rows a warp walks
    (both buffers and both barrier phases reused).  Every other shape here (k >= 35, or rows shorter than 512 steps)
    takes dw_tc_kernel, whose zero-filled TMA boxes supply the halos and the clip tail.  Also: garbage in the pitch
    padding, and 300 repeats (dw_tc_kernel, k = 59) that must be bit-identical (the mbarrier protocol is not visible to
    racecheck)."""
    shapes = [(3, 16, 1027, 35), (11, 8, 2049, 59), (2, 8, 5, 19), (2, 8, 1, 5), (9, 24, 3001, 27), (2, 16, 1024, 51),
              (17, 8, 1029, 11), (2, 16, 1030, 51), (2, 8, 9, 59), (5, 8, 756, 19), (3, 8, 748, 43),
              # short rows -> dw_tc_kernel (TMA boxes of 64 steps x up to 128 utterances): one to three 128-step tiles,
              # a batch that is not a multiple of 16 (the MMA's N rounding), the longest filters
              (256, 16, 100, 29), (11, 8, 292, 65), (9, 8, 292, 33), (3, 8, 383, 83), (13, 8, 250, 5), (2, 8, 129, 11)]
    for B, C, T, k in shapes:
        x = rnd(B, C, T, seed=T + k)
        w = rnd(C, k, seed=k, scale=1.0 / math.sqrt(k)).to(dtype)
        scale, shift = torch.rand(C, device=DEV) + 0.5, torch.randn(C, device=DEV) * 0.2
        xn = ncw(x, dtype)
        xn.data[:, :, T:] = float("nan")             # pitch padding is never data: it must not leak into the outputs
        ref = F.conv1d(xn.valid().float(), w.float()[:, None, :], padding=(k - 1) // 2, groups=C)
        ref = (ref * scale[None, :, None] + shift[None, :, None]).clamp(0, 6)
        y = K.dwconv(xn, w, scale, shift, k, 1, K.ACT_RELU6)
        torch.cuda.synchronize()
        got = y.valid().float()
        assert torch.isfinite(got).all(), (B, C, T, k)
        assert rel_err(got, ref) < OUT_TOL[dtype], (B, C, T, k, rel_err(got, ref))
    B, C, T, k = 11, 8, 2049, 59
    xn = ncw(rnd(B, C, T, seed=5), dtype)
    w = rnd(C, k, seed=6, scale=0.2).to(dtype)
    shift = torch.zeros(C, device=DEV)
    first = K.dwconv(xn, w, None, shift, k, 1, K.ACT_NONE)
    n_bad = torch.zeros((), device=DEV, dtype=torch.int64)
    for _ in range(300):
        n_bad += (K.dwconv(xn, w, None, shift, k, 1, K.ACT_NONE).valid() != first.valid()).sum()
    assert int(n_bad) == 0


@pytest.mark.parametrize("dtype", DTYPES)
def test_dwconv_long_rows_and_stride2(dtype):
    B, C, T, k = 2, 16, 3001, 83                       # 60 s clip: 24 dw_tc_kernel tiles of 128 steps per row
    x = rnd(B, C, T, seed=9)
    w = rnd(C, k, seed=10, scale=0.1).to(dtype)
    shift = torch.zeros(C, device=DEV)
    xn = ncw(x, dtype)
    y = K.dwconv(xn, w, None, shift, k, 1, K.ACT_NONE)
    ref = F.conv1d(xn.valid().float(), w.float()[:, None, :], padding=41, groups=C)
    assert rel_err(y.valid().float(), ref) < OUT_TOL[dtype]
    B, C, T, k = 3, 256, 1501, 11                      # asr layer 0: stride 2
    x = rnd(B, C, T, seed=11)
    w = rnd(C, k, seed=12, scale=0.3).to(dtype)
    xn = ncw(x, dtype)
    y = K.dwconv(xn, w, None, torch.zeros(C, device=DEV), k, 2, K.ACT_RELU6)
    ref = F.conv1d(xn.valid().float(), w.float()[:, None, :], stride=2, padding=5, groups=C).clamp(0, 6)
    assert y.T == 751 == ref.shape[2]
    assert rel_err(y.valid().float(), ref) < OUT_TOL[dtype]
    for simt in (False, True):                         # the any-shape kernel agrees too
        y2 = K.dwconv(xn, w, None, torch.zeros(C, device=DEV), k, 2, K.ACT_RELU6, simt=simt)
        assert rel_err(y2.valid().float(), ref) < OUT_TOL[dtype]


@pytest.mark.parametrize("k", [3, 5, 11, 19, 31, 59, 61])
@pytest.mark.parametrize("T", [1501, 100, 2600, 1])
@pytest.mark.parametrize("dtype", DTYPES)
def test_dwconv_stride2_polyphase_matches_torch(k, T, dtype):
    """Stride 2 as two polyphase stride-1 FIRs on the tensor cores (k <= 59; 61 takes the CUDA-core kernel), vs fp32
    F.conv1d(stride=2) on the same operands and vs the any-shape kernel: odd/even T, rows longer than one 1024-output
    chunk, a ragged channel count, more batch rows than one warp walks."""
    B, C = 11, 20
    x = rnd(B, C, T, seed=51)
    w = rnd(C, k, seed=52, scale=1.0 / math.sqrt(k)).to(dtype)
    scale, shift = torch.rand(C, device=DEV) + 0.5, rnd(C, seed=53)
    xn = ncw(x, dtype)
    ref = F.conv1d(xn.valid().float(), w.float()[:, None, :], stride=2, padding=(k - 1) // 2, groups=C)
    ref = (ref * scale[None, :, None] + shift[None, :, None]).clamp(0, 6)
    y = K.dwconv(xn, w, scale, shift, k, 2, K.ACT_RELU6)
    assert y.T == (T - 1) // 2 + 1 == ref.shape[2]
    assert rel_err(y.valid().float(), ref) < OUT_TOL[dtype]
    y2 = K.dwconv(xn, w, scale, shift, k, 2, K.ACT_RELU6, simt=True)
    assert rel_err(y2.valid().float(), ref) < OUT_TOL[dtype]
    y3 = K.dwconv(xn, w, None, shift, k, 2, K.ACT_NONE)                  # no scale, no activation
    ref3 = F.conv1d(xn.valid().float(), w.float()[:, None, :], stride=2, padding=(k - 1) // 2, groups=C) + shift[None, :, None]
    assert rel_err(y3.valid().float(), ref3) < OUT_TOL[dtype]


# ------------------------------------------------------------------------------------------------
# log-mel
# ------------------------------------------------------------------------------------------------
def test_logmel_matches_oracle_and_golden():
    from helpers import golden
    g = golden("logmel")
    tr = MelSpectrogramAudioTransform().to(DEV)
    clips = [synth.noise_waveform(1, 16000, seed=11)[0], synth.harmonic_waveform(1, 12345, seed=12)[0],
             synth.noise_waveform(1, 400, seed=13)[0]]
    L = max(len(c) for c in clips)
    wav = np.zeros((3, L), np.float32)
    for i, c in enumerate(clips):
        wav[i, :len(c)] = c
    lengths = torch.tensor([len(c) for c in clips], dtype=torch.int32)
    audio, audio_len = tr.logmel_batch(torch.from_numpy(wav).to(DEV), lengths.to(DEV))
    torch.cuda.synchronize()
    assert audio_len.tolist() == g["batch_audio_len"].tolist()
    # fp32 FFT round-off only matters in near-silent bins of the clean harmonic clip (see oracle test)
    np.testing.assert_allclose(audio.cpu().numpy(), g["batch_audio"], rtol=0, atol=3e-3)
    np.testing.assert_allclose(audio[0].cpu().numpy(), g["noise_16000"], rtol=0, atol=2e-4)
    mp = tr.melspec(torch.from_numpy(clips[1]).to(DEV)).cpu().numpy()
    assert mp.shape == g["harm_12345_melpower"].shape
    np.testing.assert_allclose(mp, g["harm_12345_melpower"], rtol=2e-3, atol=1e-6)
    one = tr(torch.from_numpy(clips[0]).to(DEV)).cpu().numpy()
    np.testing.assert_allclose(one, g["noise_16000"], rtol=0, atol=2e-4)


def test_logmel_ragged_batch_bf16_ncw():
    tr = MelSpectrogramAudioTransform().to(DEV)
    B, L = 9, 16000 * 3 + 77
    wav = torch.from_numpy(synth.noise_waveform(B, L, seed=5))
    lengths = torch.from_numpy(synth.ragged_lengths(B, 300, L, seed=5))
    ref, ref_len = orc.logmel_batch(wav, lengths.tolist())
    out, out_len = tr.logmel_batch(wav.to(DEV), lengths.to(DEV), ncw_bf16=True)
    torch.cuda.synchronize()
    assert out_len.cpu().tolist() == ref_len.tolist()
    got = out.valid().float().transpose(1, 2).cpu()
    assert got.shape == ref.shape
    # bf16 has 8 mantissa bits: |x| < 16 -> abs error <= 2^-5
    assert float((got - ref).abs().max()) <= 0.0625 + 1e-3
    assert (got[0, int(ref_len[0]):] == torch.tensor(orc.BLANK_AUDIO).to(torch.bfloat16).float()).all()


def test_logmel_int16_pcm_equals_fp32():
    """int16 PCM input scaled by 1/32768 in the kernel == fp32 samples s/32768 (what torchaudio.load returns for a
    16-bit WAV, data_modules.py:288): bit-identical features in every output mode, half the input bytes."""
    tr = MelSpectrogramAudioTransform().to(DEV)
    B, L = 5, 16000 * 2 + 123
    g = torch.Generator().manual_seed(6)
    pcm = torch.randint(-32768, 32768, (B, L), generator=g, dtype=torch.int32).to(torch.int16)
    pcm[1] = (pcm[1].float() * 0.01).to(torch.int16)                       # a quiet clip
    wav = pcm.float() / 32768.0
    lengths = torch.tensor([L, L - 777, 5000, L - 1, 300], dtype=torch.int32)
    a32, n32 = tr.logmel_batch(wav.to(DEV), lengths.to(DEV))
    a16, n16 = tr.logmel_batch(pcm.to(DEV), lengths.to(DEV))
    assert torch.equal(a32, a16) and torch.equal(n32, n16) and n16.tolist() == [1 + int(n) // 160 for n in lengths]
    b32, _ = tr.logmel_batch(wav.to(DEV), lengths.to(DEV), ncw_dtype=torch.bfloat16)
    b16, _ = tr.logmel_batch(pcm.to(DEV), lengths.to(DEV), ncw_dtype=torch.bfloat16)
    assert torch.equal(b32.valid(), b16.valid())
    ref, _ = orc.logmel_batch(wav, lengths.tolist())
    np.testing.assert_allclose(a16.cpu().numpy(), ref.numpy(), rtol=0, atol=3e-3)
    assert torch.equal(tr.melspec(pcm[0].to(DEV)), tr.melspec(wav[0].to(DEV)))
    # an odd row pitch (rows not 4-byte aligned for int16): the scalar load path gives the same features
    odd = torch.zeros((B, L + 1), dtype=torch.int16)
    odd[:, :L] = pcm
    c16, _ = tr.logmel_batch(odd.to(DEV)[:, :L + 1], lengths.to(DEV))
    assert torch.equal(c16[:, : a16.shape[1]], a16)


def test_logmel_short_and_empty_clips_are_safe():
    """torchaudio refuses clips of <= n_fft/2 samples (reflect padding).  Device-resident lengths cannot be checked
    without a sync, so the kernel must stay in bounds: lengths are clamped to [0, L_max], the reflected index is
    clamped into the clip, an empty slot yields BLANK_AUDIO only (the filler slots of a fixed-shape graph batch).
    Host-resident lengths are validated and raise."""
    from voice100_b200 import V100Error
    tr = MelSpectrogramAudioTransform().to(DEV)
    L = 4000
    big = torch.randn(6, L, device=DEV) * 0.1
    wav = big[1:5]                                                     # neighbours on both sides would be read by a bug
    lengths = torch.tensor([0, 1, 256, 10 ** 6], dtype=torch.int32, device=DEV)
    audio, audio_len = tr.logmel_batch(wav, lengths)
    torch.cuda.synchronize()
    assert torch.isfinite(audio).all()
    assert audio_len.tolist() == [1, 1, 2, 1 + L // 160]               # 1 + len // 160 with len clamped to L_max
    assert (audio[0] == orc.BLANK_AUDIO).all() and (audio[1, 1:] == orc.BLANK_AUDIO).all()
    full, _ = tr.logmel_batch(wav, torch.tensor([L] * 4, dtype=torch.int32, device=DEV))
    assert torch.equal(audio[3], full[3])                              # the over-long length was clamped to the row
    ref = orc.logmel_clip(wav[3].cpu())
    np.testing.assert_allclose(audio[3].cpu().numpy(), ref.numpy(), rtol=0, atol=3e-3)
    for bad in ([L, 200, L, L], [L, L, L + 1, L]):
        with pytest.raises(V100Error):
            tr.logmel_batch(wav, torch.tensor(bad, dtype=torch.int32))
    tr.logmel_batch(wav, torch.tensor([L, 0, 257, L], dtype=torch.int32))   # 0 = empty slot, 257 = shortest legal clip
    with pytest.raises(V100Error):
        tr.melspec(wav[0, :256])


# ------------------------------------------------------------------------------------------------
# small layout / head kernels
# ------------------------------------------------------------------------------------------------
def test_layout_and_head_kernels():
    x = rnd(3, 101, 64, seed=20)
    z = rnd(2, 40, 77, seed=21)
    for dtype in DTYPES:
        y = K.ntc_f32_to_ncw(x, dtype)
        assert torch.equal(y.valid().float(), x.transpose(1, 2).to(dtype).float())
        assert torch.equal(K.ncw_to_f32(K.ncw_from_f32(z, dtype)), z.to(dtype).float())
    ids = torch.randint(0, 29, (3, 45), device=DEV)
    table = rnd(29, 64, seed=22).to(torch.bfloat16)
    e = K.embedding_ncw(ids, table)
    assert torch.equal(e.valid(), F.embedding(ids, table).transpose(1, 2))
    # the shared-memory gather at model shapes (8 channel blocks, ragged last group, partial channel block) and the
    # global-memory fallback for a table too large to stage
    for (Be, Te, Ve, Ce) in ((5, 292, 29, 512), (2, 100, 71, 24), (3, 7, 44, 72), (2, 33, 1000, 64)):
        ids_e = torch.randint(0, Ve, (Be, Te), device=DEV)
        for dtype in DTYPES:
            tab_e = rnd(Ve, Ce, seed=Ve).to(dtype)
            assert torch.equal(K.embedding_ncw(ids_e, tab_e).valid(), F.embedding(ids_e, tab_e).transpose(1, 2))
    lg = K.Ncw(torch.randn(4, 29, 104, device=DEV), 101)
    lg.data[0, 3, 7] = lg.data[0, 11, 7] = 50.0          # tie -> first maximal index
    logits, tokens = K.ctc_finalize(lg)
    ref = lg.valid().transpose(1, 2)
    assert torch.equal(logits, ref) and torch.equal(tokens, ref.argmax(-1)) and int(tokens[0, 7]) == 3
    assert torch.equal(K.ncw_f32_to_ntc(lg), ref)
    w = K.Ncw(torch.randn(2, 260, 56, device=DEV), 53)
    mean, std = torch.randn(259, device=DEV), torch.rand(259, device=DEV) + 0.5
    hasf0, f0, logspc, codeap = K.world_finalize(w, mean, std, True)
    v = w.valid()
    assert torch.equal(hasf0, v[:, 0])
    ref_f0 = torch.where(v[:, 0] < 0, torch.zeros(1, device=DEV), std[0] * v[:, 1] + mean[0])
    torch.testing.assert_close(f0, ref_f0, rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(logspc, (std[1:258, None] * v[:, 2:259] + mean[1:258, None]).transpose(1, 2), rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(codeap, (std[258] * v[:, 259:] + mean[258]).transpose(1, 2), rtol=1e-6, atol=1e-6)
    h2, f2, l2, c2 = K.world_finalize(w, None, None, False)
    assert torch.equal(f2, v[:, 1]) and torch.equal(l2, v[:, 2:259].transpose(1, 2))
    # output_length emitted by the CTC tail (asr.py:81-82)
    alen = torch.tensor([101, 100, 1, 0], dtype=torch.int32, device=DEV)
    _, tok2, olen = K.ctc_finalize(lg, False, alen)
    assert torch.equal(tok2, tokens) and olen.tolist() == [51, 50, 1, 0] and olen.dtype == torch.int32
    # ids outside the table: IndexError like nn.Embedding (and the flag is cleared for the next call)
    bad = ids.clone()
    bad[1, 4] = 29
    with pytest.raises(IndexError):
        K.embedding_ncw(bad, table)
    bad[1, 4] = -1
    with pytest.raises(IndexError):
        K.embedding_ncw(bad, table)
    assert torch.equal(K.embedding_ncw(ids, table).valid(), e.valid())


@pytest.mark.parametrize("S,A,layout", [(257, 1, 1), (25, 1, 1), (257, 1, 2), (25, 1, 2), (25, 3, 2), (40, 2, 1)])
def test_world_finalize_layouts(S, A, layout):
    """v1 layout [hasf0|f0|logspc(S)|codeap(A)] (tts.py:181-200) and v2 layout with the hascodeap gate
    (_tts_v2.py:65-91), S = 257 bins or 25 mel-cepstra, against the reference's split / unnormalize / where."""
    B, T = 3, 77
    C = 2 + S + (2 if layout == 2 else 1) * A
    y = K.Ncw(torch.randn(B, C, 80, device=DEV), T)
    mean, std = torch.randn(1 + S + A, device=DEV), torch.rand(1 + S + A, device=DEV) + 0.5
    x = y.valid().transpose(1, 2)                                   # [B, T, C] as the reference sees it
    sizes = [1, 1, S, A] if layout == 1 else [1, 1, S, A, A]
    parts = torch.split(x, sizes, dim=2)
    out = K.world_finalize(y, None, None, False, S, A, layout)
    assert torch.equal(out[0], parts[0][:, :, 0]) and torch.equal(out[1], parts[1][:, :, 0])
    for got, ref in zip(out[2:], parts[2:]):
        assert torch.equal(got, ref)
    out = K.world_finalize(y, mean, std, True, S, A, layout)
    f0 = torch.where(parts[0][:, :, 0] < 0, torch.zeros(1, device=DEV), std[0] * parts[1][:, :, 0] + mean[0])
    logspc = std[1:1 + S] * parts[2] + mean[1:1 + S]
    codeap = std[1 + S:] * parts[-1] + mean[1 + S:]
    if layout == 2:
        codeap = torch.where(parts[3] < 0, torch.zeros(1, device=DEV), codeap)
    torch.testing.assert_close(out[1], f0, rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(out[2], logspc, rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(out[-1], codeap, rtol=1e-6, atol=1e-6)
    assert ((out[1] == 0) == (parts[0][:, :, 0] < 0)).all()


def test_ctc_collapse_matches_reference_text_rule():
    from voice100_b200.text import CharTokenizer
    tok = CharTokenizer()
    g = torch.Generator().manual_seed(3)
    B, T = 37, 101
    # runs of repeated ids with blanks in between, like greedy CTC output
    base = torch.randint(0, 29, (B, T), generator=g)
    rep = torch.randint(0, 3, (B, T), generator=g)
    tokens = torch.where(rep > 0, torch.roll(base, 1, dims=1), base)
    tokens[:, ::7] = 0
    valid = torch.randint(0, T + 1, (B,), generator=g)
    valid[0], valid[1] = 0, T
    ids, counts = K.ctc_collapse(tokens.to(DEV), valid.to(DEV))
    torch.cuda.synchronize()
    for b in range(B):
        seq = tokens[b, : int(valid[b])].tolist()
        text = tok.decode(seq)
        ref = tok.merge_repeated(text)
        got = tok.decode(ids[b, : int(counts[b])].tolist())
        # merge_repeated additionally maps the single string " " to "" (text.py:102-103); ids keep the space
        assert got == ref or (ref == "" and got == " "), (b, text, ref, got)
        assert (ids[b, int(counts[b]):] == 0).all()


def test_ctc_best_path_matches_oracle_bit_exact():
    """Integer/index work: the device Viterbi must reproduce the reference DP exactly (golden + live oracle)."""
    import voice100_b200 as v
    from helpers import golden
    g = golden("viterbi")
    cases = [(int(T), int(L)) for T, L in g["cases"]]
    extra = [(300, 60, 900), (751, 200, 901), (97, 48, 902), (20, 30, 903)]      # last: too few frames
    T_max = max([c[0] for c in cases] + [e[0] for e in extra])
    L_max = max([c[1] for c in cases] + [e[1] for e in extra])
    B = len(cases) + len(extra)
    lp = torch.zeros(B, T_max, 29)
    text = torch.zeros(B, L_max, dtype=torch.int64)
    n_frames, n_text, refs = [], [], []
    for ci, (T, L) in enumerate(cases):
        a, lab = synth.viterbi_inputs(T, L, 29, int(g["seed"]) + ci)
        refs.append(None if int(g[f"c{ci}_fail"]) else (g[f"c{ci}_score"], g[f"c{ci}_path"], g[f"c{ci}_labels"]))
        lp[ci, :T], text[ci, :L] = torch.from_numpy(a), torch.from_numpy(lab)
        n_frames.append(T); n_text.append(L)
    for ei, (T, L, seed) in enumerate(extra):
        a, lab = synth.viterbi_inputs(T, L, 29, seed)
        try:
            refs.append(orc.ctc_best_path(a, lab))
        except IndexError:
            refs.append(None)
        lp[len(cases) + ei, :T], text[len(cases) + ei, :L] = torch.from_numpy(a), torch.from_numpy(lab)
        n_frames.append(T); n_text.append(L)
    score, hist, path, _ = v.ctc_best_path_batch(lp.to(DEV), torch.tensor(n_frames), text.to(DEV), torch.tensor(n_text))
    torch.cuda.synchronize()
    for b, ref in enumerate(refs):
        T = n_frames[b]
        if ref is None:
            assert torch.isnan(score[b]) and (hist[b] == -1).all()
            continue
        assert float(score[b]) == float(np.float32(ref[0])), b
        assert np.array_equal(hist[b, :T].cpu().numpy(), ref[1]) and np.array_equal(path[b, :T].cpu().numpy(), ref[2]), b
        assert (hist[b, T:] == 0).all()
    assert refs[-1] is None
    # raw logits in, log_softmax folded into the kernel (_asr_v2.py:95): same paths, scores to fp32 round-off
    logits = (lp * 3.0 + torch.randn(B, T_max, 1)).to(DEV)              # any per-frame shift: log_softmax removes it
    s2, h2, p2, _ = v.ctc_best_path_batch(logits, torch.tensor(n_frames), text.to(DEV), torch.tensor(n_text), normalize=True)
    s3, h3, p3, _ = v.ctc_best_path_batch(torch.log_softmax(logits, -1), torch.tensor(n_frames), text.to(DEV), torch.tensor(n_text))
    ok = ~torch.isnan(s3)
    assert torch.equal(torch.isnan(s2), torch.isnan(s3))
    torch.testing.assert_close(s2[ok], s3[ok], rtol=2e-5, atol=1e-3)
    agree = (h2[ok] == h3[ok]).float().mean()
    assert agree > 0.999, agree                                         # (a 1-ulp tie may move a boundary by a frame)
    # a label outside [0, V): IndexError for host-resident text, NaN / -1 for that utterance when it lives on the device
    bad = text.clone()
    bad[1, 2] = 29
    with pytest.raises(IndexError):
        v.ctc_best_path_batch(lp.to(DEV), torch.tensor(n_frames), bad, torch.tensor(n_text))
    s4, h4, _, _ = v.ctc_best_path_batch(lp.to(DEV), torch.tensor(n_frames), bad.to(DEV), torch.tensor(n_text))
    assert torch.isnan(s4[1]) and (h4[1] == -1).all() and float(s4[0]) == float(score[0]) and torch.equal(h4[0], hist[0])


def test_logmel_generic_configs_match_reference_golden():
    """MelSpectrogramAudioTransform with constructor arguments other than 512 / 400 / 160 / 64 (v100_logmel_generic) against
    the reference class built with the same arguments (tests/golden/logmel_generic.npz), single clips and a ragged batch,
    fp32 and int16 PCM input.  Same tolerances as the tuned kernel: 2e-4 absolute on the log-mel values of the noise clip,
    3e-3 on the clean harmonic clip (fp32 FFT round-off in its near-silent bins)."""
    import voice100_b200 as v
    from helpers import golden
    g = golden("logmel_generic")
    clips = {"noise": synth.noise_waveform(1, 6000, seed=111)[0], "harm": synth.harmonic_waveform(1, 4321, seed=112)[0]}
    i = 0
    while f"c{i}_cfg" in g.files:
        sr, n_fft, win, hop, n_mels = [int(x) for x in g[f"c{i}_cfg"]]
        tr = v.MelSpectrogramAudioTransform(sr, n_fft, win, hop, n_mels).to(DEV)
        assert tr.audio_size == n_mels
        for name, w in clips.items():
            ref = g[f"c{i}_{name}"]
            got = tr(torch.from_numpy(w).to(DEV)).cpu().numpy()
            assert got.shape == ref.shape
            err = float(np.abs(got - ref).max())
            # (fp32 FFT round-off only matters in the near-silent bins of the clean harmonic clip, as for the tuned kernel)
            assert err < (2e-4 if name == "noise" else 3e-3), (i, name, err)
        # ragged batch: [noise, harm padded], NTC fp32 and NCW bf16, frames past a clip's own length are BLANK_AUDIO
        L = 6000
        wav = np.zeros((2, L), np.float32)
        wav[0] = clips["noise"]; wav[1, :4321] = clips["harm"]
        lens = torch.tensor([6000, 4321], dtype=torch.int32)
        audio, audio_len = tr.logmel_batch(torch.from_numpy(wav).to(DEV), lens.to(DEV))
        assert audio_len.tolist() == [1 + 6000 // hop, 1 + 4321 // hop] and audio.shape == (2, 1 + L // hop, n_mels)
        n1 = 1 + 4321 // hop
        assert np.abs(audio[1, :n1].cpu().numpy() - g[f"c{i}_harm"]).max() < 3e-3
        assert bool((audio[1, n1:] == v.BLANK_AUDIO).all())
        ncw, _ = tr.logmel_batch(torch.from_numpy(wav).to(DEV), lens.to(DEV), ncw_dtype=torch.bfloat16)
        assert ncw.C == n_mels and float((ncw.valid().float().transpose(1, 2) - audio).abs().max()) < 0.07   # bf16 rounding at |x| <= 16
        pcm = torch.from_numpy(np.round(wav * 32767.0).astype(np.int16))
        a16, _ = tr.logmel_batch(pcm.to(DEV), lens.to(DEV))
        a32, _ = tr.logmel_batch((pcm.float() / 32768.0).to(DEV), lens.to(DEV))
        assert float((a16 - a32).abs().max()) < 1e-4
        i += 1
    assert i == 4
    with pytest.raises(v.V100Error):
        v.MelSpectrogramAudioTransform(16000, 500, 400, 160, 64)      # n_fft must be a power of two


def test_maskaudio_matches_reference_golden_and_oracle():
    """v100_maskaudio vs the reference method's own output (tests/golden/maskaudio.npz) and vs the oracle on a larger ragged
    batch.  Tolerance 2e-6 absolute on valid frames (expf -> logf round trip, values in [-14.8, 12]); padded frames and
    floored values are BLANK_AUDIO exactly."""
    import voice100_b200 as v
    from helpers import golden
    g = golden("maskaudio")
    B, T, C, seed = [int(x) for x in g["cfg"]]
    rng = np.random.Generator(np.random.PCG64(seed))
    audio = rng.uniform(v.BLANK_AUDIO - 1.0, 12.0, size=(B, T, C)).astype(np.float32)
    audio[0, :3] = v.BLANK_AUDIO
    lens = torch.from_numpy(g["audio_len"])
    out = v.maskaudio(torch.from_numpy(audio).to(DEV), lens.to(DEV)).cpu().numpy()
    assert np.abs(out - g["out"]).max() < 2e-6
    for b, n in enumerate(g["audio_len"]):
        assert np.all(out[b, int(n):] == np.float32(v.BLANK_AUDIO))
    B, T = 67, 1501
    a = torch.from_numpy(rng.uniform(-16.0, 12.0, size=(B, T, 64)).astype(np.float32))
    ln = torch.from_numpy(rng.integers(0, T + 1, size=B).astype(np.int64))     # host lengths, int64: converted by the wrapper
    got = v.maskaudio(a.to(DEV), ln).cpu()
    ref = orc.maskaudio(a, ln)
    assert float((got - ref).abs().max()) < 2e-6
    assert torch.equal(got == v.BLANK_AUDIO, ref == v.BLANK_AUDIO)
    with pytest.raises(v.V100Error):
        v.maskaudio(a[0].to(DEV), ln[:1])                                      # not [B, T, C]


def test_errors_are_loud():
    from voice100_b200 import V100Error
    x = K.empty_ncw(1, 60, 16, DEV)     # C_in not a multiple of 8
    with pytest.raises(V100Error):
        K.conv1x1(x, torch.zeros(8, 60, device=DEV, dtype=torch.bfloat16), None, torch.zeros(8, device=DEV), 0)
    with pytest.raises(V100Error):
        K.dwconv(K.empty_ncw(1, 8, 16, DEV), torch.zeros(8, 4, device=DEV, dtype=torch.bfloat16), None,
                 torch.zeros(8, device=DEV), 4, 1, 0)
