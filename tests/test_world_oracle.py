"""Known answers for oracle/world.py, the float64 restatement of WORLD's DecodeAperiodicity and Synthesis that the
device vocoder (v100_world_synthesize) is tested against.  These pin the restatement's own conventions -- knot
intervals, pulse spacing, the minimum-phase construction, the DC removal and the fractional shift -- so that a change
to the restatement shows up here and not only as a device mismatch.  No GPU needed."""
import numpy as np
import pytest

import world as W


def test_decode_aperiodicity_knots():
    ca = np.array([[-10.0], [-0.2], [-35.0]])
    ap = W.decode_aperiodicity(ca)
    assert ap.shape == (3, 257)
    for t in (0, 2):
        assert ap[t, 0] == pytest.approx(10 ** (-60 / 20), rel=1e-12)
        assert ap[t, 96] == pytest.approx(10 ** (ca[t, 0] / 20), rel=1e-12)       # 96 * 31.25 Hz = 3000 Hz
        assert ap[t, 256] == pytest.approx(1.0, abs=1e-12)
        assert np.all(np.diff(ap[t, :97]) > 0) and np.all(np.diff(ap[t, 96:]) > 0)
    assert np.all(ap[1] == 1.0 - W.EPS)                                          # mean coded value > -0.5


def test_interp1_intervals():
    x = np.array([0.0, 1.0, 3.0])
    y = np.array([0.0, 10.0, 30.0])
    # on a knot: the interval that starts there; past the last knot: the last interval, extrapolated
    got = W.interp1(x, y, np.array([0.0, 1.0, 2.0, 3.0, 4.0]))
    assert got.tolist() == [0.0, 10.0, 20.0, 30.0, 40.0]


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_min_phase_magnitude_and_causality(seed):
    g = np.random.default_rng(seed)
    k = np.arange(257)
    a = g.uniform(-0.4, 0.4, 4)       # a smooth envelope: a few low-quefrency cosines (a short real cepstrum)
    L = -2.0 + sum(a[m] * np.cos(np.pi * (m + 1) * k / 256.0) for m in range(4))
    H = W.min_phase(L)
    assert np.allclose(np.abs(H), np.exp(L), rtol=1e-12, atol=0)
    h = np.fft.irfft(H, 512)
    assert np.sum(h[256:] ** 2) < 1e-10 * np.sum(h ** 2)
    # any L: the magnitude still holds
    Lr = g.normal(0, 3, 257)
    assert np.allclose(np.abs(W.min_phase(Lr)), np.exp(Lr), rtol=1e-12, atol=0)


def long_run_f0():
    f0 = np.zeros(40)
    f0[7:18] = 32.26
    return f0


def _spacings(f0_value, T=100):
    tb = W.timebase(np.full(T, f0_value))
    return np.diff(tb["pulse"]), tb


@pytest.mark.parametrize("f0", [80.0, 123.4, 200.0, 300.0])
def test_timebase_constant_voiced(f0):
    d, tb = _spacings(f0)
    period = W.FS / f0
    allowed = {int(np.floor(period)), int(np.ceil(period))}
    if period == int(period):
        # an integral period puts the wrap of the accumulated phase within rounding of a sample: either side of it
        allowed |= {int(period) - 1, int(period) + 1}
    assert set(d.tolist()) <= allowed
    assert d.mean() == pytest.approx(period, rel=2e-3)
    assert np.all(tb["vuv"] == 1)
    assert np.all(tb["noise_size"][:-1] == d) and tb["noise_size"][-1] == 0
    assert np.all(tb["noise_offset"] == tb["pulse"] - tb["pulse"][0])
    assert np.all((tb["tau"] > 0) & (tb["tau"] <= 1.0 / W.FS))


@pytest.mark.parametrize("f0", [0.0, 20.0, 32.2, -50.0])
def test_timebase_unvoiced_runs_at_500_hz(f0):
    d, tb = _spacings(f0)
    assert set(d.tolist()) <= {31, 32, 33} and d.mean() == pytest.approx(32.0, rel=1e-3)   # 16000 / 500, integral
    assert np.all(tb["vuv"] == 0)


def test_timebase_extrapolated_last_segment():
    # f0c[T] = 2 f0c[T-1] - f0c[T-2]: a rising contour keeps rising in the last 10 ms
    T = 20
    f0 = np.linspace(100.0, 290.0, T)
    tb = W.timebase(f0)
    last = tb["pulse"][tb["pulse"] >= 160 * (T - 1)]
    ext = 2 * f0[-1] - f0[-2]
    assert np.diff(last).min() <= int(np.ceil(W.FS / f0[-1]))
    assert np.diff(last).min() >= int(np.floor(W.FS / ext))
    # voiced -> unvoiced at the end: the extrapolated voicing is -1, so the last segment turns unvoiced halfway
    f0b = np.full(T, 150.0)
    f0b[-1] = 0.0
    tb2 = W.timebase(f0b)
    assert tb2["vuv"][tb2["pulse"] >= 160 * (T - 1) + 90].sum() == 0
    with pytest.raises(ValueError):
        W.timebase(np.array([100.0]))


def test_timebase_long_noise_run():
    # voiced f0 just above the 32.25 Hz floor next to unvoiced frames: the voiced half of the transition runs at
    # 16-32 Hz, so the run between two pulses gets longer than fft_size (a sustained voiced f0 cannot: its period is
    # at most 496 samples)
    tb = W.timebase(long_run_f0())
    assert tb["noise_size"].max() > W.N
    z = W.pulse_noise(W.noise(20000), 0, 700)
    seg = W.noise(700)
    assert np.array_equal(z, (seg - seg.mean())[:512])


@pytest.mark.parametrize("shift", [0.0, 0.25, 0.5, 0.75])
def test_periodic_response_flat_spectrum(shift):
    """sp = 1, ap at its 0.001 floor: h is a fractionally delayed impulse after DC removal."""
    S = np.ones((1, 257))
    A = np.full((1, 257), W.AP_MIN ** 2)
    h = W.periodic_response(S, A, np.array([1]), np.array([shift / W.FS]))[0]
    assert abs(h.sum()) < 1e-9 * np.abs(h).max()                                # DC removal with sum(r) = 1
    peak = int(np.argmax(h))
    if shift != 0.5:                                                             # 0.5 is a tie between the two
        assert peak == (W.N // 2 + 1 if shift > 0.5 else W.N // 2)
    e = np.sum(h ** 2) / W.N ** 2
    if shift == 0.0:
        assert e == pytest.approx(1.0, rel=0.01)
    if shift == 0.5:
        assert 0.85 < e < 0.95


def test_periodic_response_off():
    S = np.ones((2, 257))
    A = np.full((2, 257), 0.5)
    A[1, 0] = 0.9995
    h = W.periodic_response(S, A, np.array([0, 1]), np.array([0.0, 0.0]))
    assert np.all(h == 0.0)


def test_dc_remover_sums_to_one():
    r = W.dc_remover()
    assert r.sum() == pytest.approx(1.0, abs=1e-14)
    assert np.array_equal(r, r[::-1])


def test_noise_stream():
    z = W.noise(1_000_000)
    assert abs(z.mean()) < 5e-3 and abs(z.var() - 1.0) < 5e-3
    assert np.array_equal(z, W.noise(1_000_000))
    assert np.array_equal(W.noise(1000), z[:1000])
    assert np.all(np.round(z * 2 ** 28) == z * 2 ** 28)                          # multiples of 2^-28


def test_synthesize_shapes_and_rejections():
    T = 40
    f0 = np.full(T, 150.0)
    f0[20:] = 0.0
    y = W.synthesize(f0, np.full((T, 257), -4.0), np.full((T, 1), -20.0))
    assert y.shape == (160 * T,) and np.isfinite(y).all() and np.abs(y).max() > 0
    with pytest.raises(ValueError):
        W.synthesize(f0[:1], np.zeros((1, 257)), np.zeros((1, 1)))
    bad = np.full((T, 257), -4.0)
    bad[3, 7] = np.nan
    with pytest.raises(ValueError):
        W.synthesize(f0, bad, np.full((T, 1), -20.0))
    with pytest.raises(ValueError):
        W.synthesize(f0, np.zeros((T, 25)), np.full((T, 1), -20.0))
