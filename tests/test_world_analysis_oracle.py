"""Known answers of the float64 WORLD analysis restatement (oracle/world_analysis.py), the contract of
v100_world_analyze.  CPU only."""
import math
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import world as W  # noqa: E402
import world_analysis as A  # noqa: E402
from world_analysis_data import harmonic, roundtrip_metrics, roundtrip_params  # noqa: E402

L1 = 16000


def test_constants():
    assert A.N_BANDS == 7
    assert [round(b, 1) for b in A.BOUNDARY_F0] == [100.4, 142.0, 200.8, 284.0, 401.6, 568.0, 803.3]
    assert [4 * A.band_half(i) for i in range(7)] == [320, 224, 160, 112, 80, 56, 40]
    assert len(A.lowcut_taps()) == 641 and len(A.dio_taps()) == 641 + 992
    assert abs(A.lowcut_taps().sum()) < 1e-15
    assert [A.n_frames(n) for n in (0, 159, 160, 479, 480, 16000, 16159)] == [1, 1, 2, 3, 4, 101, 101]
    assert all(A.n_frames(n) == n // 160 + 1 for n in range(0, 100000, 7))
    assert abs(A.CT_F0_FLOOR - 94.30) < 0.005
    assert (A.D4C_FFT, A.D4C_WIN, A.D4C_BOUNDARY, A.D4C_CENTER) == (2048, 769, 21, 384)
    assert (A.LT_FFT, A.LT_B0, A.LT_B1, A.LT_B2) == (2048, 13, 512, 1012)
    assert A.VOICE_RANGE_MIN == 3 and A.MIN_FRAMES == 4
    # dither draws of one frame
    assert A.ct_draws(150.0) == 2 * 160 + 1 + 257 and A.ct_draws(500.0) == 2 * 48 + 1 + 257
    assert A.lovetrain_draws(0.0) == 0 and A.lovetrain_draws(150.0) == 321 and A.lovetrain_draws(30.0) == 1201
    assert A.d4c_draws(150.0) == 3 * 427 and A.d4c_draws(40.0) == 3 * 1363
    assert max(A.ct_draws(f) for f in np.linspace(94.31, 1000, 500)) <= 766


def _interior(T):
    t = np.arange(T) * 0.01
    return (t >= 0.05) & (t <= L1 / 16000 - 0.05), t


@pytest.mark.parametrize("name,f0_of_t", [("150 Hz", lambda t: 150.0 + 0 * t),
                                          ("120->240 Hz glide", lambda t: 120.0 * 2.0 ** t)])
def test_harmonic_tones(name, f0_of_t):
    """f0 within 0.5 % and voiced on every interior frame, flat or tilted.  codeap <= -20 dB holds for the tilted tone
    only (measured -57.6 dB at most): D4C analyses a frame only where LoveTrain finds more than 85 % of the 0.1-7.9 kHz
    power below 4 kHz, and a flat complex up to 7.9 kHz has half of it there (measured ratio 0.49-0.51), so its frames
    keep the unanalysed value 20 log10(1 - 1e-12), as WORLD's D4C leaves them."""
    m, t = _interior(101)
    for tilt in (None, lambda f: np.exp(-f / 2000.0)):
        r = A.encode(harmonic(L1, f0_of_t, tilt).astype(np.float32))
        assert r["status"] == A.OK and len(r["f0"]) == 101
        err = np.abs(r["f0"][m] / f0_of_t(t[m]) - 1.0)
        assert (r["f0"][m] > 0).all() and err.max() <= 0.005, (name, err.max())
        if tilt is None:
            assert (r["codeap"][m] == A.CODEAP_UNVOICED).all()
        else:
            assert r["codeap"][m].max() <= -20.0, r["codeap"][m].max()


def test_envelope_slope():
    """Harmonic amplitudes exp(-f / 2000): the power envelope's log falls by 1e-3 per Hz."""
    r = A.encode(harmonic(L1, lambda t: 150.0 + 0 * t, lambda f: np.exp(-f / 2000.0)).astype(np.float32))
    fr = np.arange(257) * 31.25
    band = (fr >= 300) & (fr <= 6000)
    m, _ = _interior(101)
    slopes = np.array([np.polyfit(fr[band], row[band], 1)[0] for row in r["logspc"][m]])
    assert np.abs(slopes / -1e-3 - 1.0).max() <= 0.05, slopes


def test_digital_silence():
    r = A.encode(np.zeros(L1, np.float32))
    assert r["status"] == A.OK and (r["f0"] == 0).all()
    assert (r["codeap"] == 20.0 * math.log10(1.0 - 1e-12)).all()
    assert np.isfinite(r["logspc"]).all()
    # the dither stream decides the envelope here: frame t reads values [off_t, off_t + draws) of WORLD's randn
    tab = W.noise(101 * A.ct_draws(500.0) + 1)
    x = np.zeros(L1)
    for t in (0, 50, 100):
        off = t * A.ct_draws(500.0)
        ref = np.log(A.cheaptrick_frame(x, t * 0.01, 500.0, tab[off:off + A.ct_draws(500.0)]) + 1e-15)
        np.testing.assert_array_equal(r["logspc"][t], ref)
        other = np.log(A.cheaptrick_frame(x, t * 0.01, 500.0, tab[off + 1:off + 1 + A.ct_draws(500.0)]) + 1e-15)
        assert np.abs(other - ref).max() > 1e-3


def test_white_noise_is_aperiodic():
    x = (0.1 * np.random.default_rng(7).standard_normal(L1)).astype(np.float32)
    r = A.encode(x)
    assert np.median(r["codeap"]) > -3.0


def test_rejected_input():
    assert A.encode(np.zeros(479, np.float32))["status"] == A.SHORT
    assert A.encode(np.zeros(480, np.float32))["status"] == A.OK
    x = np.zeros(1000, np.float32)
    x[500] = np.nan
    r = A.encode(x)
    assert r["status"] == A.NONFINITE and r["f0"].shape == (0,) and r["logspc"].shape == (0, 257)


def _cands(T, value):
    c = np.zeros((7, T))
    c[2] = value
    return c


def test_fix_f0_two_frame_island_removed():
    T = 20
    best = np.zeros(T)
    best[8:10] = 150.0
    assert (A.fix_f0_contour(best, _cands(T, 150.0)) == 0).all()


def test_fix_f0_jump_is_cut():
    T = 30
    best = np.full(T, 150.0)
    best[15:] = 150.0 * 1.15
    out = A.fix_f0_contour(best, _cands(T, 0.0))
    assert out[14] == 0.0 and out[15] == 0.0          # step 1 cuts frame 15, step 2 erodes both sides of the cut
    assert out[5] == 150.0 and out[20] == 150.0 * 1.15


def test_fix_f0_run_is_extended():
    T = 30
    best = np.zeros(T)
    best[10:20] = 200.0
    c = _cands(T, 0.0)
    c[2, 10:20] = 200.0                                 # step 2 leaves 12..18; steps 3 and 4 restore 10, 11 and 19
    c[3, 20:23] = [205.0, 230.0, 209.0]                 # 205 is within 10 % of the reference, 230 not
    c[4, 20:23] = [400.0, 400.0, 400.0]
    c[3, 8:10] = [190.0, 199.0]
    out = A.fix_f0_contour(best, c)
    assert (out[10:20] == 200.0).all() and out[20] == 205.0 and out[21] == 0.0
    assert out[9] == 199.0 and out[8] == 190.0 and out[7] == 0.0


def test_coding_matches_decode():
    for v in (-40.0, -25.0, -3.0, -0.7):
        ap = np.full((1, 257), 0.5)
        ap[0, 96] = 10.0 ** (v / 20.0)
        code = A.code_aperiodicity(ap)
        assert abs(code[0, 0] - v) < 1e-12
        assert abs(W.decode_aperiodicity(code)[0, 96] - ap[0, 96]) < 1e-12
    assert (W.decode_aperiodicity(np.array([[A.CODEAP_UNVOICED]])) == 1.0 - 1e-12).all()


def test_round_trip_restatements():
    """oracle/world.py synthesis, then this analysis, recovers the parameters (measured: f0 0.07 % / 0.05 %, voicing
    0.96 / 0.97, envelope 0.40 / 0.49 neper for seeds 0 and 1)."""
    for seed in (0, 1):
        f0, logspc, codeap = roundtrip_params(150, seed)
        r = A.encode(W.synthesize(f0, logspc, codeap).astype(np.float32))
        ferr, agree, rms = roundtrip_metrics(f0, logspc, r["f0"], r["logspc"])
        assert ferr <= 0.02 and agree >= 0.90 and rms <= 1.0, (seed, ferr, agree, rms)
