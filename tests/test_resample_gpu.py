"""v100_resample on the device: accuracy against the float64 restatement (oracle/resample.py) and torchaudio, owned
outputs, determinism and batch independence, 64-bit offsets, graph capture, the ASR pipelines' `sample_rate`, and
argument errors."""
import math

import numpy as np
import pytest
import torch

import resample as R
import v100_oracle as orc
import voice100_b200 as v
from helpers import golden
from voice100_b200 import V100Error, _lib, synth
from voice100_b200 import data_modules as dm
from voice100_b200 import kernels as K

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)

RATIOS = [(48000, 16000), (44100, 16000), (32000, 16000), (24000, 16000), (22050, 16000), (11025, 16000),
          (8000, 16000), (16000, 22050), (16000, 24000), (16000, 44100), (16000, 48000)]


def _batch(L, seed, int16):
    """Rows of noise with a ragged set of lengths (0, 1, shorter than the filter, ...) inside a wider row pitch whose
    padding is NaN (fp32) or a full-scale value (int16): padding must never reach a result."""
    g = np.random.default_rng(seed)
    lengths = [L, 0, 1, 5, L // 3, L - 1, 37]
    B, P = len(lengths), L + 29
    if int16:
        x = g.integers(-32768, 32768, (B, P)).astype(np.int16)
        pad = 32767
    else:
        x = (0.5 * g.standard_normal((B, P))).astype(np.float32)
        pad = np.nan
    for b, n in enumerate(lengths):
        x[b, n:] = pad
    return x, lengths


def _ref(x, lengths, a, b, L_out=None):
    tab = dm.resample_table(a, b, device="cpu")
    return R.resample_packed(x, lengths, tab.start.numpy(), tab.count.numpy(), tab.off.numpy(), tab.taps.numpy(),
                             tab.o, tab.n, tab.width, L_out)


@pytest.mark.parametrize("int16", [False, True])
@pytest.mark.parametrize("a,b", RATIOS)
def test_matches_restatement(a, b, int16):
    L = 3001
    x, lengths = _batch(L, a + b, int16)
    xd = torch.from_numpy(x).to(DEV)[:, :L]                      # row pitch L + 29 > L
    out, out_len = v.resample(xd, a, b, lengths=torch.tensor(lengths, dtype=torch.int32, device=DEV))
    ref, ref_len = _ref(x[:, :L], lengths, a, b)
    got = out.cpu().numpy().astype(np.float64)
    assert got.shape == ref.shape and out_len.cpu().tolist() == ref_len.tolist()
    assert np.isfinite(got).all()
    d = got - ref
    assert np.abs(d).max() <= 1e-6 * np.abs(ref).max(), (np.abs(d).max(), np.abs(ref).max())
    assert np.sqrt(np.mean(d ** 2)) <= 5e-7 * np.sqrt(np.mean(ref ** 2))
    for r, n in enumerate(ref_len):
        assert (got[r, n:] == 0).all()


@pytest.mark.parametrize("a,b", RATIOS)
def test_matches_torchaudio(a, b):
    AF = pytest.importorskip("torchaudio.functional")
    x = (0.5 * np.random.default_rng(a * b % 9973).standard_normal((3, 4410))).astype(np.float32)
    ref = AF.resample(torch.from_numpy(x), a, b).numpy()
    got = v.resample(torch.from_numpy(x).to(DEV), a, b).cpu().numpy()
    assert got.shape == ref.shape
    assert np.abs(got - ref).max() <= 2e-5 * np.abs(ref).max()
    # [..., L] shapes are kept, and the kaiser window / other parameters run the same kernel
    x3 = torch.from_numpy(x).reshape(3, 1, 4410)
    got3 = v.resample(x3.to(DEV), a, b, 16, 0.945, "sinc_interp_kaiser").cpu()
    ref3 = AF.resample(x3, a, b, 16, 0.945, "sinc_interp_kaiser")
    assert got3.shape == ref3.shape and float((got3 - ref3).abs().max()) <= 2e-5 * float(ref3.abs().max())


def test_owned_output_nan_padding_and_batch_independence():
    a, b, L = 44100, 16000, 20000
    x, lengths = _batch(L, 7, False)
    xd = torch.from_numpy(np.nan_to_num(x, nan=0.0)).to(DEV)
    xn = torch.from_numpy(x).to(DEV)                                # the same data, NaN padding
    lens = torch.tensor(lengths, dtype=torch.int32, device=DEV)
    tab = dm.resample_table(a, b, device=DEV)
    L_out = dm.resampled_length(L, a, b)
    B, pitch, guard = len(lengths), L_out + 64, 1024
    buf = torch.full((guard + B * pitch + guard,), float("nan"), device=DEV)
    out_len = torch.full((B,), -7, dtype=torch.int32, device=DEV)
    K._call(xn, "v100_resample", xn.data_ptr(), 0, lens.data_ptr(), B, xn.stride(0), L, tab.start.data_ptr(),
            tab.count.data_ptr(), tab.off.data_ptr(), tab.taps.data_ptr(), tab.taps.numel(), tab.o, tab.n, tab.width,
            buf[guard:].data_ptr(), pitch, L_out, out_len.data_ptr())
    rows = buf[guard:guard + B * pitch].view(B, pitch)
    assert not torch.isnan(rows[:, :L_out]).any()                   # every sample of every row written, no NaN read
    assert torch.isnan(rows[:, L_out:]).all() and torch.isnan(buf[:guard]).all() and torch.isnan(buf[-guard:]).all()
    ref, ref_len = v.resample(xd, a, b, lengths=lens)              # rows of L + 29: a wider output, zeros past L_out
    assert ref.shape[1] > L_out and (ref[:, L_out:] == 0).all()
    ref = ref[:, :L_out]
    assert torch.equal(rows[:, :L_out], ref) and torch.equal(out_len, ref_len)
    for r, n in enumerate(lengths):                                 # each row is its own single-utterance call
        one, one_len = v.resample(xd[r:r + 1, :max(n, 1)], a, b, lengths=lens[r:r + 1])
        m = one.shape[1] if n > 0 else 0
        assert int(one_len) == int(ref_len[r]) and torch.equal(one[0, :m], ref[r, :m])
    reps = [v.resample(xn[:, :L], a, b, lengths=lens)[0] for _ in range(100)]
    assert all(torch.equal(r, ref) for r in reps)


def test_graphed_equals_eager():
    a, b = 48000, 16000
    x, lengths = _batch(9000, 3, True)
    xd = torch.from_numpy(x).to(DEV)
    lens = torch.tensor(lengths, dtype=torch.int32, device=DEV)
    eager, eager_len = v.resample(xd, a, b, lengths=lens)          # builds the table outside capture
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        v.resample(xd, a, b, lengths=lens)
    torch.cuda.current_stream().wait_stream(s)
    with torch.cuda.graph(g):
        out, out_len = v.resample(xd, a, b, lengths=lens)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager) and torch.equal(out_len, eager_len)
    with pytest.raises(V100Error):                                 # an unbuilt table cannot be built during capture
        g2 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g2):
            v.resample(xd, 37000, 16000, lengths=lens)


def test_64bit_offsets():
    """Two int16 rows of 1.2e9 samples: the second row's samples sit past element 2^31."""
    a, b = 44100, 16000
    P = 1_200_000_000
    gen = torch.Generator(device=DEV).manual_seed(11)
    x = torch.randint(-32768, 32768, (2, P), device=DEV, dtype=torch.int16, generator=gen)
    lens = torch.tensor([1000, P - 3], dtype=torch.int32, device=DEV)
    out, out_len = v.resample(x, a, b, lengths=lens)
    n_last = int(out_len[1])
    assert n_last == dm.resampled_length(P - 3, a, b)
    tab = dm.resample_table(a, b, device="cpu")
    # restatement of a window at the end of the last row: start at frame j_s, far enough back for the filter
    j_s = (P - 3) // tab.o - 40
    seg = x[1, j_s * tab.o:P - 3].cpu().numpy()[None]
    ref, _ = R.resample_packed(seg, [seg.shape[1]], tab.start.numpy(), tab.count.numpy(), tab.off.numpy(),
                               tab.taps.numpy(), tab.o, tab.n, tab.width)
    skip = (tab.width // tab.o + 2) * tab.n                          # outputs whose filter reaches before the window
    q0 = j_s * tab.n + skip
    # out_len carries torchaudio's float32 rounding (spacing 32 at 4e8 samples); compare where both are defined
    m = min(n_last - q0, ref.shape[1] - skip)
    got = out[1, q0:q0 + m].cpu().numpy().astype(np.float64)
    want = ref[0, skip:skip + m]
    assert m > 4000
    assert np.abs(got - want).max() <= 1e-6 * np.abs(want).max()
    assert (out[1, n_last:] == 0).all()


# ---------------------------------------------------------------------------------------------- pipelines

@pytest.fixture(scope="module")
def asr_v1():
    sd = orc.to_torch_sd(synth.asr_state_dict(64, 128, 29, 128, seed=3, randomize_bn=True))
    m = v.AudioToTextCTC(64, 128, 29, 128)
    m.load_state_dict(sd)
    return v.AsrPipeline(v.MelSpectrogramAudioTransform().to(DEV), m.to(DEV).eval())


@pytest.fixture(scope="module")
def asr_v2():
    settings = synth.ASR_V2_SMALL_ENCODER
    sd = orc.to_torch_sd(synth.asr_v2_state_dict(64, settings, 2, 256, 29, seed=3, randomize_ln=True, gain=2.0))
    m = v.AudioToAlignText(64, [list(r) for r in settings], 2, 256, 29)
    m.load_state_dict(sd)
    return v.AsrV2Pipeline(v.MelSpectrogramAudioTransform().to(DEV), m.to(DEV).eval())


def _wav44k(int16):
    B, L = 5, 44100 * 2 + 17
    g = torch.Generator().manual_seed(44)
    pcm = torch.randint(-8000, 8000, (B, L), generator=g, dtype=torch.int32).to(torch.int16)
    wav = pcm if int16 else pcm.float() / 32768.0
    lengths = torch.tensor([L, L - 4410, 30000, 0, 1234], dtype=torch.int32)
    return wav, lengths


@pytest.mark.parametrize("int16", [False, True])
@pytest.mark.parametrize("version", [1, 2])
def test_pipeline_sample_rate_is_resample_then_pipeline(asr_v1, asr_v2, version, int16):
    pipe = asr_v1 if version == 1 else asr_v2
    wav, lengths = _wav44k(int16)
    wd, ld = wav.to(DEV), lengths.to(DEV)
    want = pipe(*v.resample(wd, 44100, 16000, lengths=ld))
    got = pipe(wd, ld, sample_rate=44100)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    host = pipe(wd, lengths, sample_rate=44100)                       # host lengths: validated after resampling
    assert torch.equal(host[0], want[0]) and torch.equal(host[1], want[1])
    ids = pipe.transcribe_ids(wd, ld, sample_rate=44100)
    ids_ref = pipe.transcribe_ids(*v.resample(wd, 44100, 16000, lengths=ld))
    assert torch.equal(ids[0], ids_ref[0]) and torch.equal(ids[1], ids_ref[1])
    run = pipe.graphed(wav.shape[0], wav.shape[1], DEV, wav.dtype, sample_rate=44100)
    tok, ol = run(wd, ld)
    torch.cuda.synchronize()
    assert torch.equal(tok, want[0]) and torch.equal(ol, want[1])
    tok_h, len_h = pipe.transcribe_host(wav.pin_memory(), lengths.pin_memory(), device=DEV, chunks=2, sample_rate=44100)
    assert torch.equal(tok_h, want[0].cpu()) and torch.equal(len_h, want[1].cpu())
    # the native rate: None, 16000 and no keyword are the same call
    w16, l16 = v.resample(wd, 44100, 16000, lengths=ld)
    base = pipe(w16, l16)
    for sr in (None, 16000):
        o = pipe(w16, l16, sample_rate=sr)
        assert torch.equal(o[0], base[0]) and torch.equal(o[1], base[1])
    run16 = pipe.graphed(w16.shape[0], w16.shape[1], DEV, sample_rate=16000)
    assert torch.equal(run16(w16, l16)[0], base[0])


def test_logmel_of_44k_clip_matches_golden():
    gd = golden("resample")
    tr = v.MelSpectrogramAudioTransform().to(DEV)
    clip = torch.from_numpy(gd["clip44k"]).to(DEV)
    ref = gd["clip44k_logmel"]
    audio, audio_len = tr.logmel_batch(clip[None], torch.tensor([clip.shape[0]], dtype=torch.int32), orig_freq=44100)
    assert audio.shape[1] == ref.shape[0] and int(audio_len[0]) == ref.shape[0]
    np.testing.assert_allclose(audio[0].cpu().numpy(), ref, rtol=0, atol=3e-3)
    one = tr(clip.float() / 32768.0, orig_freq=44100).cpu().numpy()
    np.testing.assert_allclose(one, ref, rtol=0, atol=3e-3)
    rs = v.resample(clip, 44100, 16000).cpu().numpy()
    ta = gd["clip44k_resampled"]
    assert rs.shape == ta.shape and np.abs(rs - ta).max() <= 2e-5 * np.abs(ta).max()
    with pytest.raises(V100Error):                                   # resampled length 37: too short for n_fft / 2
        tr.logmel_batch(clip[None], torch.tensor([100], dtype=torch.int32), orig_freq=44100)


def test_errors_launch_nothing():
    x = torch.zeros((2, 1000), device=DEV)
    lens = torch.tensor([1000, 10], dtype=torch.int32, device=DEV)
    v.resample(x, 44100, 16000, lengths=lens)                          # tables built, library loaded
    n0 = _lib.stats["launches"]
    with pytest.raises(ValueError):
        v.resample(x, -44100, 16000)
    with pytest.raises(Exception, match="integer"):
        v.resample(x, 44100.5, 16000)
    with pytest.raises(ValueError):
        v.resample(x, 44100, 16000, lowpass_filter_width=0)
    with pytest.raises(ValueError):
        v.resample(x, 44100, 16000, resampling_method="sinc_interp_linear")
    with pytest.raises(V100Error):
        v.resample(x.double(), 44100, 16000)                            # float64 is not a supported input
    with pytest.raises(V100Error):
        v.resample(x, 44100, 16000, lengths=lens[:1])                   # lengths do not match the batch
    with pytest.raises(V100Error):
        v.resample(x, 1, 20000)                                         # 20000 phases > 16384
    with pytest.raises(V100Error):
        v.resample(x, 100003, 1)                                        # input span of 4 frames > 16384 samples
    tab = dm.resample_table(44100, 16000, device=DEV)
    out = torch.empty((2, 400), device=DEV)
    args = (tab.start.data_ptr(), tab.count.data_ptr(), tab.off.data_ptr(), tab.taps.data_ptr(), tab.taps.numel(),
            tab.o, tab.n, tab.width, out.data_ptr())
    with pytest.raises(V100Error):                                      # L_out >= 2^31
        K._call(x, "v100_resample", x.data_ptr(), 0, lens.data_ptr(), 2, 1000, 1000, *args, 2 ** 31, 2 ** 31, None)
    with pytest.raises(V100Error):                                      # row pitch below the row length
        K._call(x, "v100_resample", x.data_ptr(), 0, lens.data_ptr(), 2, 999, 1000, *args, 400, 400, None)
    with pytest.raises(V100Error):                                      # unknown sample type
        K._call(x, "v100_resample", x.data_ptr(), 2, lens.data_ptr(), 2, 1000, 1000, *args, 400, 400, None)
    torch.cuda.synchronize()
    assert _lib.stats["launches"] == n0
