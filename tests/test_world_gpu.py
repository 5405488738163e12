"""WORLD synthesis on the device (v100_world_noise / _timebase / _synthesize, kernels.world_synthesize, WORLDVocoder and
the pipelines' waveform path) against the float64 restatement oracle/world.py.

The noise table and the time base are exact (bit patterns); the waveform, computed in fp32, is held to
rms(diff) <= 1e-4 rms(y) and max|diff| <= 1e-3 max|y| per utterance.  Parity of the restatement with pyworld itself is
not checked anywhere (DESIGN.md 3.8)."""
import numpy as np
import pytest
import torch

import voice100_b200 as v
import world as W
from voice100_b200 import _lib, kernels as K, synth

pytestmark = pytest.mark.gpu
DEV = "cuda"
V = 29
RMS_BAR, MAX_BAR = 1e-4, 1e-3


def _rng(seed):
    return np.random.Generator(np.random.PCG64(seed))


def world_params(B, T, seed):
    """Seeded WORLD parameters: smooth voiced contours of 80-300 Hz with unvoiced gaps, smooth log spectra that fall
    with frequency, coded aperiodicity on both sides of -0.5.  Utterance 0 has a voiced run just above the 32.25 Hz
    floor next to unvoiced frames (noise runs longer than 512), 1 negative f0, 2 logspc frames at -80 and +20."""
    g = _rng(seed)
    t = np.arange(T)[None, :]
    f0 = 190 + 110 * np.sin(2 * np.pi * t / g.uniform(40, 120, (B, 1)) + g.uniform(0, 6.3, (B, 1)))
    for b in range(B):
        for _ in range(3):
            s = int(g.integers(0, T))
            f0[b, s:s + int(g.integers(3, 20))] = 0.0
    k = np.arange(257)[None, None, :]
    logspc = (-3.0 - 6.0 * k / 256.0 + 1.5 * np.cos(2 * np.pi * k / g.uniform(60, 140, (B, 1, 1)) + 0.05 * t[..., None])
              + 0.3 * g.standard_normal((B, T, 1)))
    codeap = np.minimum(-1.0, -20.0 + 8.0 * np.sin(t / 7.0 + g.uniform(0, 6.3, (B, 1))))[..., None]
    codeap[:, ::9] = -0.3                                                        # fully aperiodic frames
    codeap[:, 4::11] = -0.6
    if B > 0 and T >= 40:
        f0[0, :] = 0.0
        f0[0, 7:18] = 32.26
    if B > 1:
        f0[1, 10:14] = -50.0
        f0[1, T - 5:] = np.linspace(200.0, 40.0, 5)                              # extrapolated knot below zero
    if B > 2:
        logspc[2, 5:9] = -80.0
        logspc[2, 12:15] = 20.0
    return f0.astype(np.float32), logspc.astype(np.float32), codeap.astype(np.float32)


def _dev(*xs):
    return [torch.from_numpy(np.ascontiguousarray(x)).to(DEV) for x in xs]


def _errors(got, ref):
    d = got.astype(np.float64) - ref
    rms_y, max_y = np.sqrt(np.mean(ref ** 2)), np.abs(ref).max()
    return float(np.sqrt(np.mean(d ** 2)) / rms_y), float(np.abs(d).max() / max_y)


# ------------------------------------------------------------------------------------------------ noise table

def test_noise_table_is_the_restatement_bit_for_bit():
    n = 70000
    got = torch.empty(n, dtype=torch.float64, device=DEV)
    _lib.call("v100_world_noise", got.data_ptr(), n, torch.cuda.current_stream().cuda_stream)
    assert np.array_equal(got.cpu().numpy().view(np.int64), W.noise(n).view(np.int64))
    cached = K.world_noise(n, DEV)
    assert cached.numel() >= n and torch.equal(cached[:n], got)


# ------------------------------------------------------------------------------------------------ time base

def test_timebase_exact():
    B, T = 12, 160
    f0, logspc, codeap = world_params(B, T, seed=11)
    frame_len = np.array([T, 2, 3, T - 1, 57, T, 100, 41, T, 8, 121, T], np.int32)
    f0_d, sp_d, ap_d, fl_d = _dev(f0, logspc, codeap, frame_len)
    tb = K.world_timebase(f0_d, sp_d, ap_d, fl_d)
    head, info, tau = tb["head"].cpu().numpy(), tb["info"].cpu().numpy(), tb["tau"].cpu().numpy()
    assert (tb["status"].cpu().numpy() == K.WORLD_OK).all()
    long_runs = 0
    for b in range(B):
        n = int(frame_len[b])
        ref = W.timebase(f0[b, :n].astype(np.float64))
        y_len = ref["y_len"]
        assert int(head[b, 1]) == y_len == int(tb["wav_len"][b])
        pulses = np.nonzero(info[b, :y_len] >= 0)[0]
        assert np.array_equal(pulses, ref["pulse"]), b
        assert int(head[b, 3]) == len(pulses) and int(head[b, 2]) == (pulses[0] if len(pulses) else 0)
        assert np.array_equal(info[b, pulses] & 1, ref["vuv"]), b
        assert np.array_equal(info[b, pulses] >> 1, ref["noise_size"]), b
        assert np.array_equal(tau[b, pulses].view(np.int64), ref["tau"].view(np.int64)), b
        long_runs += int((ref["noise_size"] > W.N).sum())
    assert long_runs > 0                                                         # the > 512 noise rule is exercised


# ------------------------------------------------------------------------------------------------ waveform

def test_waveform_matches_restatement():
    B, T = 6, 150
    f0, logspc, codeap = world_params(B, T, seed=21)
    frame_len = np.array([T, 2, 3, T, 77, 131], np.int32)
    wav, wav_len, status = K.world_synthesize(*_dev(f0, logspc, codeap, frame_len))
    wav, wav_len = wav.cpu().numpy(), wav_len.cpu().numpy()
    assert (status.cpu().numpy() == K.WORLD_OK).all()
    report = []
    for b in range(B):
        n = int(frame_len[b])
        ref = W.synthesize(f0[b, :n], logspc[b, :n], codeap[b, :n])
        assert int(wav_len[b]) == len(ref)
        e_rms, e_max = _errors(wav[b, :len(ref)], ref)
        report.append((b, n, e_rms, e_max))
        assert e_rms <= RMS_BAR and e_max <= MAX_BAR, (b, e_rms, e_max)
        assert (wav[b, len(ref):] == 0).all()
    print("world waveform vs restatement (utterance, frames, rms/rms, max/max):", report)


def test_owned_output_and_guards():
    """Direct C call into a NaN-filled buffer with guard bands and a pitch wider than 160 T."""
    B, T = 5, 90
    f0, logspc, codeap = world_params(B, T, seed=31)
    frame_len = np.array([T, 40, 2, 1, 63], np.int32)
    f0_d, sp_d, ap_d, fl_d = _dev(f0, logspc, codeap, frame_len)
    pitch, G = 160 * T + 333, 4096
    buf = torch.full((B * pitch + 2 * G,), float("nan"), device=DEV)
    buf[:G] = 1234.5
    buf[-G:] = -1234.5
    wav = buf[G:G + B * pitch]
    out = torch.full((2, B), -7, dtype=torch.int32, device=DEV)
    noise = K.world_noise(160 * T, DEV)
    ws = K._world_workspace(B, T, DEV)
    _lib.call("v100_world_synthesize", *K._world_args(f0_d, sp_d, ap_d, fl_d), B, T, noise.data_ptr(), noise.numel(),
              ws.data_ptr(), wav.data_ptr(), pitch, out[0].data_ptr(), out[1].data_ptr(),
              torch.cuda.current_stream().cuda_stream)
    host = buf.cpu().numpy()
    assert (host[:G] == 1234.5).all() and (host[-G:] == -1234.5).all()
    rows = host[G:G + B * pitch].reshape(B, pitch)
    wl = out[0].cpu().numpy()
    assert wl.tolist() == [160 * T, 160 * 40, 320, 0, 160 * 63]
    assert out[1].cpu().tolist() == [0, 0, 0, K.WORLD_SHORT, 0]
    for b in range(B):
        assert np.isfinite(rows[b, :wl[b]]).all() and (rows[b, wl[b]:] == 0).all(), b
    ref, _, _ = K.world_synthesize(f0_d, sp_d, ap_d, fl_d)
    assert torch.equal(torch.from_numpy(rows[:, :160 * T].copy()), ref.cpu())


def test_status_rejects_and_spares_the_rest():
    B, T = 5, 60
    f0, logspc, codeap = world_params(B, T, seed=41)
    frame_len = np.array([T, 1, T, 30, T], np.int32)
    clean = K.world_synthesize(*_dev(f0, logspc, codeap, frame_len))
    f0b, spb, apb = f0.copy(), logspc.copy(), codeap.copy()
    spb[2, 17, 100] = np.nan
    f0b[3, 45] = np.nan                   # past utterance 3's 30 frames: not used, not rejected
    apb[4, 0, 0] = np.inf
    wav, wav_len, status = K.world_synthesize(*_dev(f0b, spb, apb, frame_len))
    assert status.cpu().tolist() == [K.WORLD_OK, K.WORLD_SHORT, K.WORLD_NONFINITE, K.WORLD_OK, K.WORLD_NONFINITE]
    assert wav_len.cpu().tolist() == [160 * T, 0, 0, 160 * 30, 0]
    assert (wav[[1, 2, 4]] == 0).all()
    for b in (0, 3):
        assert torch.equal(wav[b], clean[0][b])
    f0n = f0.copy()
    f0n[0, 5] = np.nan
    st = K.world_synthesize(*_dev(f0n, logspc, codeap, frame_len))[2]
    assert int(st[0]) == K.WORLD_NONFINITE
    one = K.world_synthesize(*_dev(f0[:, :1], logspc[:, :1], codeap[:, :1]))
    assert (one[2] == K.WORLD_SHORT).all() and (one[1] == 0).all() and (one[0] == 0).all()


def test_deterministic_and_batch_independent():
    B, T = 8, 120
    f0, logspc, codeap = world_params(B, T, seed=51)
    frame_len = np.array([T, 60, 3, T, 99, 2, T, 110], np.int32)
    args = _dev(f0, logspc, codeap, frame_len)
    first = K.world_synthesize(*args)[0]
    for _ in range(100):
        assert torch.equal(K.world_synthesize(*args)[0], first)
    for b in range(B):
        alone = K.world_synthesize(args[0][b:b + 1], args[1][b:b + 1], args[2][b:b + 1], args[3][b:b + 1])[0]
        assert torch.equal(alone[0], first[b]), b


def test_strided_inputs_read_in_place():
    B, T = 3, 70
    f0, logspc, codeap = world_params(B, T, seed=55)
    ref = K.world_synthesize(*_dev(f0, logspc, codeap))[0]
    big = torch.zeros((B, T, 300), device=DEV)
    big[:, :, 3:260] = torch.from_numpy(logspc).to(DEV)
    big[:, :, 1] = torch.from_numpy(f0).to(DEV)
    big[:, :, 280] = torch.from_numpy(codeap[..., 0]).to(DEV)
    got = K.world_synthesize(big[:, :, 1], big[:, :, 3:260], big[:, :, 280:281])[0]
    assert torch.equal(got, ref)


def test_vocoder_interface():
    with pytest.raises(v.V100Error):
        v.WORLDVocoder(sample_rate=22050)
    with pytest.raises(v.V100Error):
        v.WORLDVocoder(n_fft=1024)
    voc = v.WORLDVocoder()
    f0, logspc, codeap = world_params(3, 80, seed=61)
    wav, wav_len, _ = voc.decode_batch(*_dev(f0, logspc, codeap))
    for b in range(3):
        y = voc.decode(f0[b], logspc[b], codeap[b])
        assert y.dtype == np.float64 and y.shape == (160 * 80,)
        assert np.array_equal(y, wav[b, :int(wav_len[b])].double().cpu().numpy())
    with pytest.raises(ValueError):
        voc.decode(f0[0, :1], logspc[0, :1], codeap[0, :1])
    with pytest.raises(v.V100Error):
        voc.decode_batch(*_dev(f0, logspc[..., :25].copy(), codeap))


# ------------------------------------------------------------------------------------------------ pipelines

def _load(model, sd):
    model.load_state_dict({k: torch.from_numpy(np.asarray(t)) for k, t in sd.items()})
    return model.to(DEV).eval()


def _realistic_head(sd, key, scale=0.1):
    sd = dict(sd)
    sd[key + ".weight"] = (np.asarray(sd[key + ".weight"]) * scale).astype(np.float32)
    sd[key + ".bias"] = np.log1p(np.array([0.5, 2.0], np.float32)).astype(np.float32)
    return sd


@pytest.fixture(scope="module")
def tts_v1():
    H = 512
    amodel = _load(v.TextToAlignTextModel(V, H), _realistic_head(synth.align_state_dict(V, H, seed=1234), "layers.4"))
    vmodel = _load(v.AlignTextToAudioModel(V, H), synth.audio_state_dict(V, H, seed=1234))
    return v.TtsPipeline(amodel, vmodel)


@pytest.fixture(scope="module")
def tts_v2():
    amodel = _load(v.TextToAlignText(V, 2, 256, 2), _realistic_head(synth.align_v2_state_dict(V, 2, 256, 2, seed=62),
                                                                    "dense"))
    dec = [list(r) for r in synth.TTS_V2_BASE_DECODER]
    mcep = _load(v.AlignTextToAudio(V, 25, 1, 2, 512, dec), synth.audio_v2_state_dict(V, 25, seed=63))
    return amodel, mcep


def test_v1_waveform_is_decode_of_the_pipeline(tts_v1):
    """The bench-sized v1 batch (256 x 100 tokens): waveform == decode_batch(pipe(...)) bit for bit, and three sampled
    utterances against the restatement."""
    B, L = 256, 100
    text = torch.from_numpy(synth.text_tokens(B, L, V, seed=2024)).to(DEV)
    f0, logspc, codeap, frame_len, _ = tts_v1(text)
    wav, wav_len, status = tts_v1.waveform(text)
    ref = v.WORLDVocoder().decode_batch(f0, logspc, codeap, frame_len)
    assert torch.equal(wav, ref[0]) and torch.equal(wav_len, ref[1]) and torch.equal(status, ref[2])
    assert (status == K.WORLD_OK).all() and torch.equal(wav_len, 160 * frame_len)
    report = []
    for b in (0, 101, 255):
        n = int(frame_len[b])
        y = W.synthesize(f0[b, :n].cpu().numpy(), logspc[b, :n].cpu().numpy(), codeap[b, :n].cpu().numpy())
        e_rms, e_max = _errors(wav[b, :len(y)].cpu().numpy(), y)
        report.append((b, n, e_rms, e_max))
        assert e_rms <= RMS_BAR and e_max <= MAX_BAR, (b, e_rms, e_max)
    print("v1 256 x 100 pipeline, sampled utterances vs restatement:", report)


def test_v2_waveform_with_mcep_model(tts_v2):
    amodel, mcep = tts_v2
    pipe = v.TtsV2Pipeline(amodel, v.AlignTextToAudioPredict(mcep).to(DEV))
    B, L = 16, 60
    text = torch.from_numpy(synth.text_tokens(B, L, V, seed=77)).to(DEV)
    text_len = torch.from_numpy(_rng(78).integers(1, L + 1, B)).to(torch.int32).to(DEV)
    f0, logspc, codeap, frame_len, _ = pipe(text, text_len)
    wav, wav_len, status = pipe.waveform(text, text_len)
    ref = v.WORLDVocoder().decode_batch(f0, logspc, codeap, frame_len)
    assert torch.equal(wav, ref[0]) and torch.equal(wav_len, ref[1]) and torch.equal(status, ref[2])
    with pytest.raises(v.V100Error, match="AlignTextToAudioPredict"):
        v.TtsV2Pipeline(amodel, mcep).waveform(text, text_len)


@pytest.mark.parametrize("version", [1, 2])
def test_graphed_waveform_matches_eager(tts_v1, tts_v2, version):
    if version == 1:
        pipe, max_frames = tts_v1, 240
    else:
        pipe, max_frames = v.TtsV2Pipeline(tts_v2[0], v.AlignTextToAudioPredict(tts_v2[1]).to(DEV)), 200
    B, L = 24, 80
    run = pipe.graphed(B, L, max_frames, waveform=True)
    default = pipe.graphed(B, L, max_frames)
    for seed in (101, 102):
        text = torch.from_numpy(synth.text_tokens(B, L, V, seed=seed)).to(DEV)
        text_len = torch.from_numpy(_rng(seed).integers(1, L + 1, B)).to(torch.int32).to(DEV)
        got = [t.clone() for t in run(text, text_len)]
        ref = pipe.waveform(text, text_len, max_frames)
        assert len(got) == 3 and all(torch.equal(g_, r_) for g_, r_ in zip(got, ref))
        assert len(default(text, text_len)) == 5
