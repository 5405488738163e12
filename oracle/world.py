"""WORLD waveform synthesis, restated in float64 numpy: the contract of v100_world_synthesize (csrc/world.cu).

This restates WORLD's `DecodeAperiodicity` (codec.cpp) and `Synthesis` (synthesis.cpp), the C++ code that
`pyworld.decode_aperiodicity` / `pyworld.synthesize` wrap and that the reference's `WORLDVocoder.decode`
(voice100/vocoder.py:89-102) calls.  It was written from a description of that code, not from its source, and has NOT
been compared with pyworld: the places where a misremembered detail would change the output are listed in DESIGN.md
(section 3.8).  Constants: fs = 16000, fft_size = 512, frame period 10 ms.

Choices written down here:
  - logspc -> sp = exp(logspc); no 1e-15 log offset is subtracted (the effect would be below 1e-15 absolute).
  - the noise is WORLD's `randn` (xorshift128, 12 uniform draws summed) restarted at every call, so one table indexed
    from the first pulse serves every utterance.
  - a pulse whose noise run is longer than fft_size keeps its first fft_size values after the mean of all of them is
    removed (WORLD writes past its buffer there; this is what its FFT reads if that overflow corrupts nothing).
"""
from __future__ import annotations

import functools

import numpy as np

FS = 16000
N = 512
FRAME_PERIOD = 10.0                    # ms
PI = 3.1415926535897932384
EPS = 1e-12                            # world::kMySafeGuardMinimum
LOWEST_F0 = FS / N + 1.0               # 32.25 Hz
DEFAULT_F0 = 500.0
AP_MIN, AP_MAX = 0.001, 0.999999999999


# ---------------------------------------------------------------------------------------------- noise (WORLD randn)

@functools.lru_cache(maxsize=4)
def _noise_cached(n: int) -> np.ndarray:
    x, y, z, w = 123456789, 362436069, 521288629, 88675123
    m = 0xFFFFFFFF
    out = np.empty(n, np.float64)
    for j in range(n):
        s = 0
        for _ in range(12):
            t = (x ^ (x << 11)) & m
            x, y, z = y, z, w
            w = (w ^ (w >> 19)) ^ (t ^ (t >> 8))
            s += w >> 4
        out[j] = s / 268435456.0 - 6.0
    out.flags.writeable = False
    return out


def noise(n: int) -> np.ndarray:
    """The first n values of WORLD's randn() stream after its reseed: xorshift128 with state (123456789, 362436069,
    521288629, 88675123); each value sums (w >> 4) over 12 steps and returns sum / 2^28 - 6 (exact in float64)."""
    if n <= 0:
        return np.zeros(0, np.float64)
    return _noise_cached(-(-int(n) // 65536) * 65536)[:n]


# ---------------------------------------------------------------------------------------------- interpolation

def interp1(x: np.ndarray, y: np.ndarray, xi: np.ndarray) -> np.ndarray:
    """WORLD's interp1 / histc: interval k holds x[k] <= xi < x[k+1]; a point on a knot takes the interval that starts
    there, points at or past the last knot take the last interval (and extrapolate), points below the first the first.
    s = (xi - x[k]) / h[k], y = y[k] + s * (y[k+1] - y[k]), h[k] = x[k+1] - x[k], each step rounded on its own."""
    x = np.asarray(x, np.float64)
    y = np.asarray(y, np.float64)
    k = np.clip(np.searchsorted(x, xi, side="right") - 1, 0, len(x) - 2)
    h = x[1:] - x[:-1]
    s = (xi - x[k]) / h[k]
    return y[k] + s * (y[k + 1] - y[k])


# ---------------------------------------------------------------------------------------------- DecodeAperiodicity

def decode_aperiodicity(codeap: np.ndarray, fs: int = FS, fft_size: int = N) -> np.ndarray:
    """codeap [T, 1] (dB) -> aperiodicity [T, fft_size/2 + 1].  A frame whose mean coded value is > -0.5 is fully
    aperiodic (1 - eps everywhere); otherwise the knots (0 Hz, -60), (3000 Hz, codeap), (fs/2, -eps) are linearly
    interpolated in dB at f_k = k fs / fft_size and converted with 10^(v/20)."""
    codeap = np.asarray(codeap, np.float64)
    if codeap.ndim != 2 or codeap.shape[1] != 1:
        raise ValueError(f"codeap must be [T, 1] at 16 kHz, got {codeap.shape}")
    bins = fft_size // 2 + 1
    freq = np.arange(bins) * float(fs) / fft_size
    knots = np.array([0.0, 3000.0, fs / 2.0])
    out = np.empty((codeap.shape[0], bins), np.float64)
    for t in range(codeap.shape[0]):
        if codeap[t].mean() > -0.5:
            out[t] = 1.0 - EPS
        else:
            v = interp1(knots, np.array([-60.0, codeap[t, 0], -EPS]), freq)
            out[t] = 10.0 ** (v / 20.0)
    return out


# ---------------------------------------------------------------------------------------------- time base

def timebase(f0: np.ndarray, fs: int = FS, frame_period: float = FRAME_PERIOD) -> dict:
    """WORLD's GetTimeBase + GetPulseLocationsForTimeBase for T >= 2 frames of f0.
    -> dict(y_len, pulse (int64 sample of each pulse), tau (fractional shift, s), vuv (0/1 at the pulse),
            noise_size, noise_offset)."""
    f0 = np.asarray(f0, np.float64)
    T = f0.shape[0]
    if T < 2:
        raise ValueError("WORLD synthesis needs at least two f0 frames")
    y_len = int(T * frame_period * fs / 1000)
    period = frame_period / 1000.0
    f0c = np.where(f0 < LOWEST_F0, 0.0, f0)
    vuv = np.where(f0c == 0.0, 0.0, 1.0)
    f0c = np.append(f0c, f0c[T - 1] * 2 - f0c[T - 2])
    vuv = np.append(vuv, vuv[T - 1] * 2 - vuv[T - 2])
    knots = np.arange(T + 1) * period
    xi = np.arange(y_len) / float(fs)
    f0i = interp1(knots, f0c, xi)
    vuvi = interp1(knots, vuv, xi)
    vuvi = np.where(vuvi > 0.5, 1.0, 0.0)
    f0i = np.where(vuvi == 0.0, DEFAULT_F0, f0i)
    phase = np.cumsum(((2.0 * PI) * f0i) / fs)          # sequential float64 sum
    w = np.fmod(phase, 2.0 * PI)
    hit = np.abs(w[1:] - w[:-1]) > PI
    pulse = np.nonzero(hit)[0]
    y1 = w[pulse] - 2.0 * PI
    y2 = w[pulse + 1]
    x = -y1 / (y2 - y1)
    tau = x / fs
    nsz = np.zeros(len(pulse), np.int64)
    if len(pulse):
        nsz[:-1] = pulse[1:] - pulse[:-1]
    off = pulse - (pulse[0] if len(pulse) else 0)
    return dict(y_len=y_len, pulse=pulse.astype(np.int64), tau=tau, vuv=vuvi[pulse].astype(np.int64),
                noise_size=nsz, noise_offset=off.astype(np.int64))


# ---------------------------------------------------------------------------------------------- per-pulse spectra

def min_phase(L: np.ndarray) -> np.ndarray:
    """Minimum-phase spectrum of the log amplitude L [..., N/2 + 1]: mirror to N points, real cepstrum (inverse DFT),
    fold (c[0], 2c[1..N/2-1], c[N/2], zeros), H = exp(DFT) with e^{-2 pi i k n / N}, bins 0..N/2."""
    L = np.asarray(L, np.float64)
    n = 2 * (L.shape[-1] - 1)
    full = np.concatenate([L, L[..., -2:0:-1]], axis=-1)
    c = np.fft.ifft(full, axis=-1).real
    fold = np.zeros(n)
    fold[0] = 1.0
    fold[1:n // 2] = 2.0
    fold[n // 2] = 1.0
    return np.exp(np.fft.fft(c * fold, axis=-1)[..., :n // 2 + 1])


def dc_remover(fft_size: int = N) -> np.ndarray:
    """r[n] = 0.5 - 0.5 cos(2 pi (n + 1) / (N + 1)) for n < N/2, mirrored, scaled to sum 1."""
    h = fft_size // 2
    r = np.empty(fft_size)
    i = np.arange(h)
    r[:h] = 0.5 - 0.5 * np.cos(2.0 * PI * (i + 1.0) / (1.0 + fft_size))
    r[fft_size - 1 - i] = r[:h]
    dc = 2.0 * r[:h].sum()
    r[:h] /= dc
    r[fft_size - 1 - i] = r[:h]
    return r


def periodic_response(S: np.ndarray, A: np.ndarray, vuv, tau, fs: int = FS) -> np.ndarray:
    """Periodic part h [P, N] for P pulses (S, A [P, N/2+1], vuv [P], tau [P] in s): zero where vuv <= 0.5 or
    A[0] > 0.999; else min-phase(0.5 log(S (1 - A) + eps)), fractional delay by cos - i sqrt(1 - cos^2),
    N irfft, fftshift, DC removal."""
    S, A = np.atleast_2d(S), np.atleast_2d(A)
    vuv, tau = np.atleast_1d(vuv), np.atleast_1d(tau)
    n = 2 * (S.shape[-1] - 1)
    on = (vuv > 0.5) & (A[:, 0] <= 0.999)
    H = min_phase(np.log(S * (1.0 - A) + EPS) / 2.0)
    coef = 2.0 * PI * tau * fs / n
    c = np.cos(coef[:, None] * np.arange(n // 2 + 1)[None, :])
    H = H * (c - 1j * np.sqrt(1.0 - c * c))
    h = np.fft.fftshift(n * np.fft.irfft(H, n, axis=-1), axes=-1)
    r = dc_remover(n)
    d = h[:, n // 2:].sum(-1, keepdims=True)
    h[:, :n // 2] = -d * r[:n // 2]
    h[:, n // 2:] -= d * r[n // 2:]
    h[~on] = 0.0
    return h


def aperiodic_response(S: np.ndarray, A: np.ndarray, vuv, z: np.ndarray) -> np.ndarray:
    """Aperiodic part a [P, N]: z [P, N] the zero-mean, zero-padded noise of each pulse; H' = min-phase(0.5 log(S A +
    eps)) where vuv != 0, else min-phase(0.5 log S); a = fftshift(N irfft(H' rfft(z)))."""
    S, A = np.atleast_2d(S), np.atleast_2d(A)
    vuv = np.atleast_1d(vuv)
    n = 2 * (S.shape[-1] - 1)
    with np.errstate(divide="ignore"):
        L = np.where((vuv != 0)[:, None], np.log(S * A + EPS), np.log(S)) / 2.0
    H = min_phase(L)
    Z = np.fft.rfft(z, n, axis=-1)
    return np.fft.fftshift(n * np.fft.irfft(H * Z, n, axis=-1), axes=-1)


def pulse_noise(noise_tab: np.ndarray, offset: int, size: int, fft_size: int = N) -> np.ndarray:
    """The zero-mean noise segment of one pulse, zero-padded (or cut) to fft_size."""
    z = np.zeros(fft_size)
    if size > 0:
        seg = noise_tab[offset:offset + size]
        seg = seg - seg.mean()
        m = min(size, fft_size)
        z[:m] = seg[:m]
    return z


# ---------------------------------------------------------------------------------------------- Synthesis

def _check(f0, logspc, codeap):
    f0 = np.asarray(f0, np.float64).reshape(-1)
    logspc = np.asarray(logspc, np.float64)
    codeap = np.asarray(codeap, np.float64)
    if codeap.ndim == 1:
        codeap = codeap[:, None]
    T = f0.shape[0]
    if logspc.shape != (T, N // 2 + 1):
        raise ValueError(f"logspc must be [{T}, {N // 2 + 1}], got {logspc.shape}")
    if codeap.shape != (T, 1):
        raise ValueError(f"codeap must be [{T}, 1], got {codeap.shape}")
    if T < 2:
        raise ValueError("WORLD synthesis needs at least two frames")
    if not (np.isfinite(f0).all() and np.isfinite(logspc).all() and np.isfinite(codeap).all()):
        raise ValueError("non-finite WORLD parameters")
    return f0, logspc, codeap


def synthesize(f0, logspc, codeap, chunk: int = 4096) -> np.ndarray:
    """One utterance: f0 [T] (Hz, 0 = unvoiced), logspc [T, 257] (natural log of the power spectrum), codeap [T, 1]
    -> float64 waveform [160 T].  Raises ValueError for T < 2 or non-finite input (WORLD has no defined behaviour)."""
    f0, logspc, codeap = _check(f0, logspc, codeap)
    T = f0.shape[0]
    sp = np.exp(logspc)
    ap = decode_aperiodicity(codeap)
    tb = timebase(f0)
    y_len = tb["y_len"]
    y = np.zeros(y_len)
    P = len(tb["pulse"])
    if P == 0:
        return y
    tab = noise(int((tb["noise_offset"] + tb["noise_size"]).max()) + 1)
    apc = np.clip(ap, AP_MIN, AP_MAX)
    for s in range(0, P, chunk):
        idx = np.arange(s, min(P, s + chunk))
        pi = tb["pulse"][idx]
        q = (pi / float(FS)) / (FRAME_PERIOD / 1000.0)
        fl = np.minimum(T - 1, np.floor(q).astype(np.int64))
        ce = np.minimum(T - 1, np.ceil(q).astype(np.int64))
        w = (q - np.floor(q))[:, None]
        same = (fl == ce)[:, None]
        S = np.where(same, np.abs(sp[fl]), (1.0 - w) * np.abs(sp[fl]) + w * np.abs(sp[ce]))
        A = np.where(same, apc[fl], (1.0 - w) * apc[fl] + w * apc[ce]) ** 2
        vuv = tb["vuv"][idx]
        h = periodic_response(S, A, vuv, tb["tau"][idx])
        z = np.stack([pulse_noise(tab, int(tb["noise_offset"][i]), int(tb["noise_size"][i])) for i in idx])
        a = aperiodic_response(S, A, vuv, z)
        resp = (h * np.sqrt(tb["noise_size"][idx].astype(np.float64))[:, None] + a) / N
        for j, p in enumerate(pi):
            off = int(p) - N // 2 + 1
            lo, hi = max(0, -off), min(N, y_len - off)
            y[off + lo:off + hi] += resp[j, lo:hi]
    return y
