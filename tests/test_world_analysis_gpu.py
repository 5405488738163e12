"""WORLD analysis on the device (v100_world_analyze, WORLDVocoder.encode / encode_batch) against the float64
restatement oracle/world_analysis.py."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import world_analysis as A  # noqa: E402
from world_analysis_data import roundtrip_metrics, roundtrip_params, speechlike_batch  # noqa: E402

pytestmark = pytest.mark.gpu

LENGTHS = [48000, 481, 1000, 480, 20000]              # row 1 is all zero (digital silence)


def _dev():
    return torch.device("cuda", 0)


def _batch(dtype):
    x = speechlike_batch(LENGTHS, seed=3)
    if dtype == "int16":
        x = np.clip(np.round(x * 32768.0), -32768, 32767).astype(np.int16)
    return x


def _run(x, lengths, pitch_extra=0, T=None):
    import voice100_b200.kernels as K
    B, L = x.shape
    full = np.zeros((B, L + pitch_extra), x.dtype)
    full[:, :L] = x
    t = torch.from_numpy(full).to(_dev())[:, :L]
    return K.world_analyze(t, torch.tensor(lengths, dtype=torch.int32, device=_dev()), T)


_ref_cache = {}


def _ref(x, n):
    key = (x.dtype.str, n, x[:n].tobytes())
    if key not in _ref_cache:
        _ref_cache[key] = A.encode(x[:n])
    return _ref_cache[key]


def test_dio_taps_match_restatement():
    import voice100_b200.kernels as K
    np.testing.assert_array_equal(K.dio_taps(_dev()).cpu().numpy(), A.dio_taps())


@pytest.mark.parametrize("dtype,pitch_extra", [("fp32", 0), ("int16", 0), ("fp32", 97)])
def test_against_restatement(dtype, pitch_extra):
    x = _batch(dtype)
    f0, sp, ap, frame_len, status = (t.cpu().numpy() for t in _run(x, LENGTHS, pitch_extra))
    assert status.tolist() == [0] * len(LENGTHS)
    for b, n in enumerate(LENGTHS):
        r = _ref(x[b], n)
        T = len(r["f0"])
        assert frame_len[b] == T == n // 160 + 1
        v = r["f0"] > 0
        np.testing.assert_array_equal(f0[b, :T] > 0, v)
        if v.any():
            assert np.abs(f0[b, :T][v] / r["f0"][v] - 1).max() <= 1e-6
        assert np.abs(sp[b, :T] - r["logspc"]).max() <= 1e-4, (b, np.abs(sp[b, :T] - r["logspc"]).max())
        un = r["codeap"][:, 0] == A.CODEAP_UNVOICED
        np.testing.assert_array_equal(ap[b, :T, 0][un], np.float32(A.CODEAP_UNVOICED))
        assert np.abs(ap[b, :T, 0] - r["codeap"][:, 0]).max() <= 1e-3
        assert (f0[b, T:] == 0).all() and (sp[b, T:] == 0).all() and (ap[b, T:] == 0).all()
    assert (f0[1] == 0).all() and (f0[0] > 0).sum() > 20      # silence row unvoiced, speech row voiced


def test_owned_outputs_and_rejections():
    """NaN-prefilled outputs with guard bands: every element of the rows is written, padding rows are 0, guards are
    untouched; a short and a NaN utterance get their status and zeros and leave the other rows unchanged."""
    import voice100_b200.kernels as K
    from voice100_b200 import _lib
    x = _batch("fp32")
    bad = x.copy()
    bad[2, 100] = np.nan
    lens = list(LENGTHS)
    lens[3] = 479
    dev = _dev()
    B, L = bad.shape
    T = L // 160 + 3
    G = 64
    wav = torch.from_numpy(bad).to(dev)
    ln = torch.tensor(lens, dtype=torch.int32, device=dev)
    bufs = [torch.full((B * T + 2 * G,), float("nan"), device=dev),
            torch.full((B * T * 257 + 2 * G,), float("nan"), device=dev),
            torch.full((B * T + 2 * G,), float("nan"), device=dev)]
    ints = torch.full((2 * B + 2 * G,), -7, dtype=torch.int32, device=dev)
    noise = K.world_noise(5290 * (L // 160 + 1), dev)
    n = int(_lib.lib().v100_world_analysis_workspace_bytes(B, L))
    ws = torch.empty((n + 256,), device=dev, dtype=torch.uint8)
    K._call(wav, "v100_world_analyze", wav.data_ptr(), 0, L, ln.data_ptr(), B, L, K.dio_taps(dev).data_ptr(),
            noise.data_ptr(), noise.numel(), ws.data_ptr() + (-ws.data_ptr()) % 256, T,
            bufs[0][G:].data_ptr(), bufs[1][G:].data_ptr(), bufs[2][G:].data_ptr(), ints[G:].data_ptr(),
            ints[G + B:].data_ptr())
    torch.cuda.synchronize()
    for buf in bufs:
        assert torch.isnan(buf[:G]).all() and torch.isnan(buf[-G:]).all() and not torch.isnan(buf[G:-G]).any()
    assert (ints[:G] == -7).all() and (ints[-G:] == -7).all()
    frame_len, status = ints[G:G + B].tolist(), ints[G + B:G + 2 * B].tolist()
    assert status == [0, 0, K.WORLD_NONFINITE, K.WORLD_SHORT, 0]
    assert frame_len[2] == frame_len[3] == 0
    f0 = bufs[0][G:-G].view(B, T)
    sp = bufs[1][G:-G].view(B, T, 257)
    ap = bufs[2][G:-G].view(B, T)
    for b in (2, 3):
        assert (f0[b] == 0).all() and (sp[b] == 0).all() and (ap[b] == 0).all()
    good = _run(x, LENGTHS)
    for b in (0, 1, 4):
        Tb = frame_len[b]
        assert torch.equal(f0[b, :Tb], good[0][b, :Tb]) and torch.equal(sp[b, :Tb], good[1][b, :Tb])
        assert torch.equal(ap[b, :Tb], good[2][b, :Tb, 0])
        assert (f0[b, Tb:] == 0).all() and (sp[b, Tb:] == 0).all() and (ap[b, Tb:] == 0).all()


def test_deterministic_and_batch_independent():
    x = _batch("fp32")
    a = _run(x, LENGTHS)
    b = _run(x, LENGTHS)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    for i in (0, 2):
        one = _run(x[i:i + 1, :LENGTHS[i]].copy(), [LENGTHS[i]])
        T = LENGTHS[i] // 160 + 1
        assert torch.equal(one[0][0, :T], a[0][i, :T]) and torch.equal(one[1][0, :T], a[1][i, :T])
        assert torch.equal(one[2][0, :T], a[2][i, :T])


def test_graph_capture_equals_eager():
    import voice100_b200 as v
    x = torch.from_numpy(_batch("fp32")).to(_dev())
    ln = torch.tensor(LENGTHS, dtype=torch.int32, device=_dev())
    voc = v.WORLDVocoder()
    eager = voc.encode_batch(x, ln)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        voc.encode_batch(x, ln)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = voc.encode_batch(x, ln)
    g.replay()
    torch.cuda.synchronize()
    for u, w in zip(eager, out):
        assert torch.equal(u, w)


@pytest.mark.parametrize("rate", [22050, 44100, 48000])
def test_other_rates_resample_first(rate):
    import voice100_b200 as v
    rng = np.random.default_rng(rate)
    lens = [rate * 2, rate // 2, 700]
    x = np.zeros((3, max(lens)), np.float32)
    for b, n in enumerate(lens):
        x[b, :n] = 0.2 * np.sin(2 * np.pi * 160 * np.arange(n) / rate) + 0.01 * rng.standard_normal(n)
    xt = torch.from_numpy(x).to(_dev())
    ln = torch.tensor(lens, dtype=torch.int32, device=_dev())
    voc = v.WORLDVocoder()
    got = voc.encode_batch(xt, ln, sample_rate=rate)
    y, yl = v.resample(xt, rate, 16000, lengths=ln)
    ref = voc.encode_batch(y, yl)
    for u, w in zip(got, ref):
        assert torch.equal(u, w)
    import voice100_b200.kernels as K
    assert got[4].tolist() == [0 if n >= 480 else K.WORLD_SHORT for n in yl.tolist()]


def test_encode_equals_batch_row():
    import voice100_b200 as v
    x = _batch("int16")
    voc = v.WORLDVocoder()
    f0, sp, ap = voc.encode(x[0, :LENGTHS[0]])
    b = voc.encode_batch(torch.from_numpy(x).to(_dev()), torch.tensor(LENGTHS, dtype=torch.int32, device=_dev()))
    T = LENGTHS[0] // 160 + 1
    assert f0.dtype == np.float64 and f0.shape == (T,) and sp.shape == (T, 257) and ap.shape == (T, 1)
    np.testing.assert_array_equal(f0, b[0][0, :T].double().cpu().numpy())
    np.testing.assert_array_equal(sp, b[1][0, :T].double().cpu().numpy())
    np.testing.assert_array_equal(ap, b[2][0, :T].double().cpu().numpy())
    with pytest.raises(ValueError):
        voc.encode(np.zeros(479, np.float32))
    bad = np.zeros(1000, np.float32)
    bad[3] = np.inf
    with pytest.raises(ValueError):
        voc.encode(bad)


def test_round_trip_synthesis_analysis():
    """world_synthesize then encode_batch recovers the WORLD parameters it was given (DESIGN 3.10 records the
    measured values)."""
    import voice100_b200 as v
    voc = v.WORLDVocoder()
    T = 300
    params = [roundtrip_params(T, seed) for seed in range(4)]
    dev = _dev()
    f0 = torch.tensor(np.stack([p[0] for p in params]), dtype=torch.float32, device=dev)
    sp = torch.tensor(np.stack([p[1] for p in params]), dtype=torch.float32, device=dev)
    ap = torch.tensor(np.stack([p[2] for p in params]), dtype=torch.float32, device=dev)
    wav, wav_len, status = voc.decode_batch(f0, sp, ap)
    ef0, esp, _, flen, est = voc.encode_batch(wav, wav_len)
    assert status.tolist() == [0] * 4 and est.tolist() == [0] * 4 and flen.tolist() == [T * 160 // 160 + 1] * 4
    res = [roundtrip_metrics(p[0], p[1], ef0[i].double().cpu().numpy(), esp[i].double().cpu().numpy())
           for i, p in enumerate(params)]
    print("round trip (f0 error, voicing agreement, envelope rms):", res)
    for ferr, agree, rms in res:
        assert ferr <= 0.02 and agree >= 0.90 and rms <= 1.0, res
