"""WORLD analysis, restated in float64 numpy: the contract of v100_world_analyze (csrc/world_analysis.cu).

This restates what the reference's `WORLDVocoder.encode` (voice100/vocoder.py:66-88) runs through pyworld:
`dio` -> `stonemask` -> `cheaptrick` -> `d4c` -> `code_aperiodicity`, then logspc = log(sp + 1e-15).  It was written
from a description of WORLD (dio.cpp, stonemask.cpp, cheaptrick.cpp, d4c.cpp, codec.cpp, common.cpp), not from its
source, and has NOT been compared with pyworld: DESIGN.md section 3.10 lists the places where a misremembered detail
would change the output.  One configuration: fs = 16000, frame period 10 ms, fft_size 512 (257 bins, one coded band).

Conventions written down here (each one a place a comparison with pyworld would have to confirm):
  DIO
  - the input loses its mean over its L samples (the mean is a fixed tree: 256 strided partial sums in sample order,
    then halved 128, 64, ... 1; `mean_fixed`), then the low-cut filter: 641-tap Hann-based high-pass h (h = -w / sum w,
    +1 at the centre tap 320), zero-phase (centre tap aligned), linear convolution with the signal zero outside [0, L).
  - band i (7 of them, boundary 71 2^((i+1)/2)): a Nuttall window of M = 4 round(fs / boundary / 2) taps (not
    normalised), delay 2 round(fs / boundary / 2): band[n] = sum_j w[j] hp[n + M/2 - j], n in [0, L).
  - both convolutions run tap by tap in ascending order, each product and sum rounded on its own (no FMA): the device
    repeats exactly these operations, so its band signals, crossings and raw f0 are bit-identical to these.
  - events: negative-going crossings of x (0 < x[e-1], x[e] <= 0), of -x, of d = x[n+1] - x[n] (peaks) and of -d
    (dips); fine edge e - x[e-1] / (x[e] - x[e-1]); intervals fs / diff at ((a + b) / 2) / fs; interp1 (histc) at the
    frame times t 10 / 1000 s.
  - a band any of whose four series has fewer than 3 intervals (4 events) gives no candidate (WORLD's
    CheckEvent(n - 2)); a candidate outside [boundary / 2, boundary] or [71, 800] is 0 with score 1e5; the score is
    the (n - 1) std of the four values over their mean; the first band with the lowest score wins.
  - FixF0Contour with voice_range_minimum 3 and allowed range 0.1: step 1 zeroes the first and last 3 frames and every
    frame with |f[i] - f[i-1]| / (1e-12 + f[i]) >= 0.1 (f the unfixed contour, so a run's first frame goes too); step 2
    zeroes every frame with an unvoiced neighbour (runs shorter than 3 vanish, longer runs lose their end frames);
    steps 3 and 4 extend each run forward from its last frame, then backward from its first, with the candidate
    (over the 7 bands) nearest to 1.5 f[j] - 0.5 f[j -/+ 1], kept while within 10 % of that reference.
  StoneMask
  - voiced frames with 40 < f0 <= fs / 12: Blackman-like window of half length int(1.5 fs / f0 + 1) around
    round((t - half / fs) fs + 0.001), sample index clamp(i - 1, 0, L - 1), time (i - 1) / fs - t; its central
    difference; FFT size 2^(2 + int(log2(2 half + 1))).  Instantaneous frequency at the harmonics round(f k N / fs):
    pass 1 with 2 harmonics (rejected: 0 if outside (0, 2 f0]), pass 2 from that estimate with
    min(int(fs / 2 / f1), 6) harmonics; a correction larger than 20 % keeps the input f0.
  CheapTrick / D4C / coding: see the functions below; the dither stream is WORLD's randn (oracle/world.py `noise`)
  restarted at every stage of every utterance; CheapTrick reads, frame by frame, 2 half + 1 values for the window,
  then 257 for the spectrum; D4C reads all LoveTrain windows first (voiced frames), then per analysed frame the two
  centroid windows and the power window.
  Input rejected (status, frame_len 0, zero rows): fewer than 4 frames (L < 480, where FixF0Contour returns early) or a
  non-finite sample.
"""
from __future__ import annotations

import math
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from world import interp1, noise  # noqa: E402

FS = 16000
N = 512
BINS = N // 2 + 1
HOP = 160
PI = 3.1415926535897932384
EPS = 1e-12                                   # world::kMySafeGuardMinimum
DBL_EPS = 2.220446049250313e-16               # world::kEps
F0_FLOOR, F0_CEIL, ALLOWED_RANGE = 71.0, 800.0, 0.1
N_BANDS = 1 + int(math.log(F0_CEIL / F0_FLOOR) / math.log(2.0) * 2.0)                 # 7
BOUNDARY_F0 = [F0_FLOOR * 2.0 ** ((i + 1) / 2.0) for i in range(N_BANDS)]
LOWCUT_HALF = int(FS / 50.0 + 0.5)                                                      # 320
VOICE_RANGE_MIN = int(0.5 + 1000.0 / 10.0 / F0_FLOOR) * 2 + 1                            # 3
CT_F0_FLOOR = 3.0 * FS / (N - 3.0)                                                      # 94.30 Hz
DEFAULT_F0 = 500.0
D4C_FFT = int(2.0 ** (1 + int(math.log(4.0 * FS / 47.0 + 1) / math.log(2.0))))          # 2048
D4C_WIN = int(3000.0 * D4C_FFT / FS) * 2 + 1                                            # 769
D4C_CENTER = int(3000.0 * D4C_FFT / FS)                                                 # 384
D4C_BOUNDARY = int(D4C_FFT * 8.0 / D4C_WIN + 0.5)                                       # 21
LT_FFT = int(2.0 ** (1 + int(math.log(3.0 * FS / 40.0 + 1) / math.log(2.0))))           # 2048
LT_B0, LT_B1, LT_B2 = (int(math.ceil(f * LT_FFT / FS)) for f in (100.0, 4000.0, 7900.0))  # 13, 512, 1012
D4C_THRESHOLD = 0.85
AP_UNVOICED = 1.0 - EPS
CODEAP_UNVOICED = 20.0 * math.log10(AP_UNVOICED)
MIN_FRAMES = VOICE_RANGE_MIN + 1                                                         # 4
OK, SHORT, NONFINITE = 0, 1, 2                                                           # V100_WORLD_*


def mround(x: float) -> int:
    """WORLD's matlab_round: halves away from zero."""
    return int(x + 0.5) if x >= 0 else int(x - 0.5)


def n_frames(L: int) -> int:
    return int(1000.0 * L / FS / 10.0) + 1


def frame_time(t):
    return np.asarray(t, np.float64) * 10.0 / 1000.0


# ---------------------------------------------------------------------------------------------- DIO

def lowcut_taps() -> np.ndarray:
    """641 taps of DIO's low-cut (50 Hz) filter, centre tap at index 320."""
    n = 2 * LOWCUT_HALF + 1
    i = np.arange(1, n + 1, dtype=np.float64)
    w = 0.5 - 0.5 * np.cos(i * 2.0 * PI / (n + 1))
    s = 0.0
    for v in w:
        s += v
    h = -w / s
    h[LOWCUT_HALF] += 1.0
    return h


def band_half(i: int) -> int:
    return mround(FS / BOUNDARY_F0[i] / 2.0)


def nuttall(n: int) -> np.ndarray:
    t = np.arange(n, dtype=np.float64) / (n - 1.0)
    return (0.355768 - 0.487396 * np.cos(2.0 * PI * t) + 0.144232 * np.cos(4.0 * PI * t)
            - 0.012604 * np.cos(6.0 * PI * t))


def dio_taps() -> np.ndarray:
    """The table the device reads: the low-cut taps, then the 7 Nuttall filters back to back (float64)."""
    return np.concatenate([lowcut_taps()] + [nuttall(4 * band_half(i)) for i in range(N_BANDS)])


def mean_fixed(x: np.ndarray) -> float:
    """Mean with a fixed summation tree (256 strided partial sums in sample order, then halved to one)."""
    L = len(x)
    pad = np.zeros(-(-L // 256) * 256)
    pad[:L] = x
    acc = np.zeros(256)
    for row in pad.reshape(-1, 256):
        acc = acc + row
    while len(acc) > 1:
        h = len(acc) // 2
        acc = acc[:h] + acc[h:]
    return float(acc[0]) / L


def dio_bands(x: np.ndarray) -> np.ndarray:
    """[7, L] band signals of DIO: mean removal, low-cut, Nuttall low-pass per band (tap by tap, no FMA)."""
    L = len(x)
    y = x - mean_fixed(x)
    h = lowcut_taps()
    H = LOWCUT_HALF
    e = 160                                            # hp is needed over [-160, L + 160)
    ypad = np.zeros(L + 2 * (H + e))
    ypad[H + e:H + e + L] = y
    n_hp = L + 2 * e
    hp = np.zeros(n_hp)                                # hp[m] is the sample at m - e
    for j in range(2 * H + 1):                         # hp[n] = sum_j h[j] y[n + H - j]
        hp = hp + h[j] * ypad[2 * H - j:2 * H - j + n_hp]
    out = np.empty((N_BANDS, L))
    for i in range(N_BANDS):
        hh = band_half(i)
        w = nuttall(4 * hh)
        acc = np.zeros(L)
        for j in range(4 * hh):                        # band[n] = sum_j w[j] hp[n + 2 hh - j]
            s = e + 2 * hh - j
            acc = acc + w[j] * hp[s:s + L]
        out[i] = acc
    return out


def fine_edges(x: np.ndarray) -> np.ndarray:
    """Refined negative-going zero crossings of x: e with 0 < x[e-1], x[e] <= 0 -> e - x[e-1] / (x[e] - x[e-1])."""
    e = np.nonzero((x[:-1] > 0.0) & (x[1:] <= 0.0))[0] + 1
    return e - x[e - 1] / (x[e] - x[e - 1])


def event_series(x: np.ndarray):
    """The four fine-edge series of one band: negative-going, positive-going, peak, dip."""
    d = (-x[:-1]) - (-x[1:])
    return [fine_edges(x), fine_edges(-x), fine_edges(d), fine_edges(-d)]


def band_candidates(x: np.ndarray, boundary: float, T: int):
    """(candidate [T], score [T]) of one band signal."""
    ser = event_series(x)
    if any(len(s) - 1 < 3 for s in ser):
        return np.zeros(T), np.full(T, 100000.0)
    tt = frame_time(np.arange(T))
    v = []
    for s in ser:
        loc = (s[:-1] + s[1:]) / 2.0 / FS
        itv = FS / (s[1:] - s[:-1])
        v.append(interp1(loc, itv, tt))
    c = (((v[0] + v[1]) + v[2]) + v[3]) / 4.0
    sd = np.sqrt(((((v[0] - c) * (v[0] - c) + (v[1] - c) * (v[1] - c)) + (v[2] - c) * (v[2] - c))
                  + (v[3] - c) * (v[3] - c)) / 3.0)
    score = sd / c
    bad = (c > boundary) | (c < boundary / 2.0) | (c > F0_CEIL) | (c < F0_FLOOR)
    return np.where(bad, 0.0, c), np.where(bad, 100000.0, score)


def select_best(cur: float, past: float, cands: np.ndarray) -> float:
    ref = (cur * 3.0 - past) / 2.0
    err = np.abs(ref - cands)
    k = int(np.argmin(err))                            # first minimum, as a strict-less scan
    best = float(cands[k])
    if abs(1.0 - best / ref) > ALLOWED_RANGE:
        return 0.0
    return best


def fix_f0_contour(best: np.ndarray, cands: np.ndarray) -> np.ndarray:
    """FixF0Contour: best [T] raw contour, cands [7, T] band candidates -> fixed contour [T]."""
    T = len(best)
    v = VOICE_RANGE_MIN
    if T <= v:
        return np.zeros(T)
    base = best.astype(np.float64).copy()
    base[:v] = 0.0
    base[T - v:] = 0.0
    s1 = np.zeros(T)
    for i in range(v, T):
        s1[i] = base[i] if abs((base[i] - base[i - 1]) / (EPS + base[i])) < ALLOWED_RANGE else 0.0
    s2 = s1.copy()
    c = (v - 1) // 2
    for i in range(c, T - c):
        if np.any(s1[i - c:i + c + 1] == 0.0):
            s2[i] = 0.0
    neg = [i - 1 for i in range(1, T) if s2[i] == 0.0 and s2[i - 1] != 0.0]
    pos = [i for i in range(1, T) if s2[i - 1] == 0.0 and s2[i] != 0.0]
    s3 = s2.copy()
    for k, start in enumerate(neg):
        limit = T - 1 if k == len(neg) - 1 else neg[k + 1]
        for j in range(start, limit):
            s3[j + 1] = select_best(s3[j], s3[j - 1], cands[:, j + 1])
            if s3[j + 1] == 0.0:
                break
    s4 = s3.copy()
    for k in range(len(pos) - 1, -1, -1):
        limit = 1 if k == 0 else pos[k - 1]
        for j in range(pos[k], limit, -1):
            s4[j - 1] = select_best(s4[j], s4[j + 1], cands[:, j - 1])
            if s4[j - 1] == 0.0:
                break
    return s4


def dio(x: np.ndarray):
    """-> (f0 [T] fixed, raw best [T], candidates [7, T])."""
    L = len(x)
    T = n_frames(L)
    bands = dio_bands(x)
    cand = np.empty((N_BANDS, T))
    score = np.empty((N_BANDS, T))
    for i in range(N_BANDS):
        cand[i], score[i] = band_candidates(bands[i], BOUNDARY_F0[i], T)
    best = np.empty(T)
    for t in range(T):
        k = 0
        for i in range(1, N_BANDS):
            if score[k, t] > score[i, t]:
                k = i
        best[t] = cand[k, t]
    return fix_f0_contour(best, cand), best, cand


# ---------------------------------------------------------------------------------------------- StoneMask

def stonemask_frame(x: np.ndarray, t: float, f0: float) -> float:
    if f0 <= 40.0 or f0 > FS / 12.0:
        return 0.0
    L = len(x)
    h = int(1.5 * FS / f0 + 1.0)
    n = 2 * h + 1
    wlen = (2.0 * h + 1.0) / FS
    nfft = int(2.0 ** (2 + int(math.log(2.0 * h + 1.0) / math.log(2.0))))
    base = mround((t + (-h) / FS) * FS + 0.001)
    raw = base + np.arange(n)
    tmp = (raw - 1.0) / FS - t
    win = 0.42 + 0.5 * np.cos(2.0 * PI * tmp / wlen) + 0.08 * np.cos(4.0 * PI * tmp / wlen)
    dwin = np.empty(n)
    dwin[0] = -win[1] / 2.0
    dwin[1:-1] = -(win[2:] - win[:-2]) / 2.0
    dwin[-1] = win[-2] / 2.0
    seg = x[np.clip(raw - 1, 0, L - 1)]
    M = np.fft.rfft(seg * win, nfft)
    D = np.fft.rfft(seg * dwin, nfft)
    num = M.real * D.imag - M.imag * D.real
    pw = M.real * M.real + M.imag * M.imag

    def fix(f, nh):
        amp = np.empty(nh)
        ifr = np.empty(nh)
        for k in range(nh):
            idx = mround(f * nfft / FS * (k + 1))
            ifr[k] = 0.0 if pw[idx] == 0.0 else idx * FS / nfft + num[idx] / pw[idx] * FS / 2.0 / PI
            amp[k] = math.sqrt(pw[idx])
        return float(np.sum(amp * ifr)) / (float(np.sum(amp * (np.arange(nh) + 1.0))) + EPS)

    f1 = fix(f0, 2)
    if f1 <= 0.0 or f1 > 2.0 * f0:
        f = 0.0
    else:
        f = fix(f1, min(int(FS / 2.0 / f1), 6))
    if abs(f - f0) > f0 * 0.2:
        f = f0
    return f


def stonemask(x: np.ndarray, f0: np.ndarray) -> np.ndarray:
    tt = frame_time(np.arange(len(f0)))
    return np.array([stonemask_frame(x, tt[i], f0[i]) for i in range(len(f0))])


# ---------------------------------------------------------------------------------------------- shared pieces

def dc_correction(p: np.ndarray, f0: float, nfft: int) -> np.ndarray:
    """WORLD's DCCorrection: bins i <= f0 N / fs gain the spectrum at f0 - f_i (interp1Q in bin units)."""
    out = p.copy()
    upper = 2 + int(f0 * nfft / FS)
    df = float(FS) / nfft
    for i in range(upper - 1):
        q = (i * FS / nfft - f0) / (-df)
        k = int(q)
        out[i] = p[i] + (p[k] + (p[k + 1] - p[k]) * (q - k))
    return out


def linear_smoothing(p: np.ndarray, width: float, nfft: int) -> np.ndarray:
    """WORLD's LinearSmoothing: mirrored ends, running sum, difference of the sum over [f - w/2, f + w/2] / w."""
    half = nfft // 2
    bnd = int(width * nfft / FS) + 1
    m = np.empty(half + 2 * bnd + 1)
    m[:bnd] = p[bnd - np.arange(bnd)]
    m[bnd:half + bnd] = p[:half]
    i = np.arange(half + bnd, half + 2 * bnd + 1)
    m[half + bnd:] = p[half - (i - (half + bnd))]
    seg = np.cumsum(m * FS / nfft)                     # sequential running sum
    df = float(FS) / nfft
    origin = -(bnd - 0.5) * FS / nfft
    fa = np.arange(half + 1) / nfft * FS - width / 2.0

    def q1(xi):
        q = (xi - origin) / df
        k = q.astype(np.int64)
        dy = np.append(seg[1:] - seg[:-1], 0.0)
        return seg[k] + dy[k] * (q - k)

    lo = q1(fa)
    hi = q1(fa + width)
    return (hi - lo) / width


def windowed(x: np.ndarray, t: float, f0: float, ratio: float, blackman: bool, dither: np.ndarray):
    """WORLD's GetWindowedWaveform (ratio periods): -> waveform [2 half + 1]; reads 2 half + 1 dither values."""
    L = len(x)
    h = mround(ratio * FS / f0 / 2.0)
    bi = np.arange(-h, h + 1)
    origin = mround(t * FS + 0.001)
    seg = x[np.clip(origin + bi, 0, L - 1)]
    pos = (2.0 * bi / ratio) / FS
    if blackman:
        w = 0.42 + 0.5 * np.cos(PI * pos * f0) + 0.08 * np.cos(PI * pos * f0 * 2)
    else:
        w = 0.5 * np.cos(PI * pos * f0) + 0.5
    wf = seg * w + dither[:2 * h + 1] * EPS
    return wf - w * (np.sum(wf) / np.sum(w))


# ---------------------------------------------------------------------------------------------- CheapTrick

def ct_draws(f0c: float) -> int:
    return 2 * mround(1.5 * FS / f0c) + 1 + BINS


def cheaptrick_frame(x: np.ndarray, t: float, f0c: float, dither: np.ndarray) -> np.ndarray:
    L = len(x)
    h = mround(1.5 * FS / f0c)
    bi = np.arange(-h, h + 1)
    origin = mround(t * FS + 0.001)
    seg = x[np.clip(origin + bi, 0, L - 1)]
    w = 0.5 * np.cos(PI * (bi / 1.5 / FS) * f0c) + 0.5
    w = w / math.sqrt(np.sum(w * w))
    wf = seg * w + dither[:2 * h + 1] * EPS
    wf = wf - w * (np.sum(wf) / np.sum(w))
    S = np.fft.rfft(wf, N)
    p = S.real * S.real + S.imag * S.imag
    p = dc_correction(p, f0c, N)
    p = linear_smoothing(p, f0c * 2.0 / 3.0, N)
    p = p + np.abs(dither[2 * h + 1:2 * h + 1 + BINS]) * DBL_EPS
    q = np.arange(1, BINS) / FS
    sl = np.ones(BINS)
    cl = np.full(BINS, (1.0 - 2.0 * (-0.15)) + 2.0 * (-0.15))
    sl[1:] = np.sin(PI * f0c * q) / (PI * f0c * q)
    cl[1:] = (1.0 - 2.0 * (-0.15)) + 2.0 * (-0.15) * np.cos(2.0 * PI * q * f0c)
    lg = np.log(p)
    cep = np.fft.rfft(np.concatenate([lg, lg[-2:0:-1]])).real        # the real cepstrum, times N
    return np.exp(np.fft.irfft(cep * sl * cl, N)[:BINS])


def cheaptrick(x: np.ndarray, f0: np.ndarray) -> np.ndarray:
    T = len(f0)
    f0c = np.where(f0 <= CT_F0_FLOOR, DEFAULT_F0, f0)
    draws = np.array([ct_draws(f) for f in f0c])
    off = np.concatenate([[0], np.cumsum(draws)])
    tab = noise(int(off[-1]))
    tt = frame_time(np.arange(T))
    return np.stack([cheaptrick_frame(x, tt[i], f0c[i], tab[off[i]:off[i + 1]]) for i in range(T)])


# ---------------------------------------------------------------------------------------------- D4C

def lovetrain_draws(f0: float) -> int:
    return 0 if f0 == 0.0 else 2 * mround(1.5 * FS / max(f0, 40.0)) + 1


def d4c_draws(f0: float) -> int:
    return 3 * (2 * mround(2.0 * FS / max(47.0, f0)) + 1)


def lovetrain_frame(x: np.ndarray, t: float, f0: float, dither: np.ndarray) -> float:
    wf = windowed(x, t, max(f0, 40.0), 3.0, True, dither)
    S = np.fft.rfft(wf, LT_FFT)
    p = S.real * S.real + S.imag * S.imag
    p[:LT_B0 + 1] = 0.0
    c = np.cumsum(p[:LT_B2 + 1])
    return float(c[LT_B1] / c[LT_B2])


def centroid(x, t, f0, dither):
    wf = np.zeros(D4C_FFT)
    w = windowed(x, t, f0, 4.0, True, dither)
    wf[:len(w)] = w
    wf[:len(w)] /= math.sqrt(np.sum(w * w))
    A = np.fft.rfft(wf)
    B = np.fft.rfft(wf * (np.arange(D4C_FFT) + 1.0))
    return B.real * A.real + A.imag * B.imag


def d4c_frame(x: np.ndarray, t: float, f0: float, dither: np.ndarray) -> float:
    """Coarse aperiodicity (dB) of the 3 kHz band for one analysed frame (f0 already max(47, f0))."""
    n = 2 * mround(2.0 * FS / f0) + 1
    sc = centroid(x, t - 0.25 / f0, f0, dither[:n]) + centroid(x, t + 0.25 / f0, f0, dither[n:2 * n])
    sc = dc_correction(sc, f0, D4C_FFT)
    S = np.fft.rfft(windowed(x, t, f0, 4.0, False, dither[2 * n:3 * n]), D4C_FFT)
    sp = S.real * S.real + S.imag * S.imag
    sp = dc_correction(sp, f0, D4C_FFT)
    sp = linear_smoothing(sp, f0, D4C_FFT)
    gd = linear_smoothing(sc / sp, f0 / 2.0, D4C_FFT)
    gd = gd - linear_smoothing(gd, f0, D4C_FFT)
    h = D4C_WIN // 2
    seg = gd[D4C_CENTER - h:D4C_CENTER + h + 1] * nuttall(D4C_WIN)
    P = np.fft.rfft(seg, D4C_FFT)
    p = np.sort(P.real * P.real + P.imag * P.imag)
    c = np.cumsum(p)
    half = D4C_FFT // 2
    v = 10.0 * math.log10(c[half - D4C_BOUNDARY - 1] / c[half])
    return min(0.0, v + (f0 - 100.0) / 50.0)


def d4c_codeap(x: np.ndarray, f0: np.ndarray):
    """-> (codeap [T, 1], LoveTrain ratios [T]); codeap = 20 log10(ap at 3000 Hz)."""
    T = len(f0)
    tt = frame_time(np.arange(T))
    lt = np.array([lovetrain_draws(f) for f in f0])
    lo = np.concatenate([[0], np.cumsum(lt)])
    ratio = np.zeros(T)
    live = np.zeros(T, bool)
    tab = noise(int(lo[-1]) + int(sum(d4c_draws(f) for f in f0 if f != 0.0)))
    for i in range(T):
        if f0[i] != 0.0:
            ratio[i] = lovetrain_frame(x, tt[i], f0[i], tab[lo[i]:lo[i + 1]])
            live[i] = ratio[i] > D4C_THRESHOLD
    code = np.full((T, 1), CODEAP_UNVOICED)
    at = int(lo[-1])
    for i in range(T):
        if not live[i]:
            continue
        fd = max(47.0, f0[i])
        n = d4c_draws(fd)
        v = d4c_frame(x, tt[i], fd, tab[at:at + n])
        at += n
        code[i, 0] = 20.0 * math.log10(10.0 ** (v / 20.0))
    return code, ratio


def code_aperiodicity(ap: np.ndarray) -> np.ndarray:
    """ap [T, 257] -> codeap [T, 1]: 20 log10(ap) at 3000 Hz (bin 96 exactly)."""
    return 20.0 * np.log10(np.asarray(ap, np.float64)[:, 96:97])


# ---------------------------------------------------------------------------------------------- encode

def as_float(wav) -> np.ndarray:
    a = np.asarray(wav)
    if a.dtype == np.int16:
        return a.astype(np.float64) / 32768.0
    return a.astype(np.float32).astype(np.float64)


def encode(wav):
    """One utterance (fp32 or int16 PCM at 16 kHz) -> dict(status, f0 [T], logspc [T, 257], codeap [T, 1]) with
    T = L // 160 + 1; a rejected utterance (SHORT: L < 480, NONFINITE) has T = 0."""
    x = as_float(wav).reshape(-1)
    L = len(x)
    empty = dict(f0=np.zeros(0), logspc=np.zeros((0, BINS)), codeap=np.zeros((0, 1)))
    if n_frames(L) < MIN_FRAMES:
        return dict(status=SHORT, **empty)
    if not np.isfinite(x).all():
        return dict(status=NONFINITE, **empty)
    f0_dio, _, _ = dio(x)
    f0 = stonemask(x, f0_dio)
    sp = cheaptrick(x, f0)
    codeap, _ = d4c_codeap(x, f0)
    return dict(status=OK, f0=f0, logspc=np.log(sp + 1e-15), codeap=codeap, f0_dio=f0_dio)
