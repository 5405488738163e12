"""Seeded signals and WORLD parameters shared by the WORLD analysis tests (CPU restatement and device)."""
from __future__ import annotations

import numpy as np

FS = 16000


def harmonic(L: int, f0_of_t, amp_of_f=None, peak: float = 0.3) -> np.ndarray:
    """Harmonic complex with instantaneous f0 f0_of_t(t) and every harmonic below 7.9 kHz (amplitude amp_of_f(f))."""
    t = np.arange(L) / FS
    f = f0_of_t(t) * np.ones(L)
    ph = 2.0 * np.pi * np.cumsum(f) / FS
    y = np.zeros(L)
    for k in range(1, int(7900 / f.min()) + 1):
        a = 1.0 if amp_of_f is None else amp_of_f(k * f)
        y += (k * f < 7900.0) * a * np.cos(k * ph)
    return peak * y / np.abs(y).max()


def speechlike(L: int, seed: int) -> np.ndarray:
    """Harmonic glides, noise bursts and digital-silence gaps."""
    rng = np.random.default_rng(seed)
    y = np.zeros(L)
    pos = 0
    while pos < L:
        n = int(rng.integers(1600, 8000))
        kind = rng.integers(0, 3)
        seg = min(n, L - pos)
        if kind == 0:
            f_a, f_b = rng.uniform(90, 280, 2)
            y[pos:pos + seg] = harmonic(seg, lambda t: f_a + (f_b - f_a) * t * FS / max(seg, 1),
                                        lambda f: np.exp(-f / 1500.0), rng.uniform(0.05, 0.5))
        elif kind == 1:
            y[pos:pos + seg] = rng.uniform(0.01, 0.2) * rng.standard_normal(seg)
        pos += seg
    return y.astype(np.float32)


def speechlike_batch(lengths, seed: int = 0):
    """[B, max(lengths) + 37] fp32 batch (padding filled with noise that must never be read) and its lengths; the
    second row is all zero."""
    rng = np.random.default_rng(seed + 1)
    L = max(lengths) + 37
    out = rng.standard_normal((len(lengths), L)).astype(np.float32)
    for b, n in enumerate(lengths):
        out[b, :n] = 0.0 if b == 1 else speechlike(n, seed + 10 * b)
    return out


def roundtrip_params(T: int, seed: int):
    """Well-behaved WORLD parameters: f0 80-300 Hz with unvoiced gaps, smooth log spectra, codeap in [-25, -1] dB."""
    rng = np.random.default_rng(seed)
    t = np.arange(T)
    f0 = 150.0 * np.exp(0.45 * np.sin(2 * np.pi * t / rng.uniform(60, 120) + rng.uniform(0, 6)))
    f0 = np.clip(f0, 80.0, 300.0)
    gap = np.zeros(T, bool)
    for s in rng.integers(10, T - 30, 3):
        gap[s:s + int(rng.integers(8, 20))] = True
    gap[:5] = gap[-5:] = True
    f0[gap] = 0.0
    k = np.arange(257)
    tilt = rng.uniform(4.0, 8.0)
    logspc = (-4.0 - tilt * k[None, :] / 256.0 + 0.8 * np.cos(k[None, :] / 24.0 + 0.05 * t[:, None])
              + 0.3 * np.sin(t[:, None] / 15.0))
    codeap = (-13.0 + 12.0 * np.sin(t / 17.0 + rng.uniform(0, 6)))[:, None]
    return f0, logspc, codeap


def roundtrip_metrics(f0, logspc, f0_est, logspc_est):
    """(median voiced-f0 relative error, voicing agreement, median rms logspc difference over 100-7000 Hz with each
    frame's mean offset removed) on frames voiced in the input and at least 3 frames from a voicing change."""
    T = min(len(f0), len(f0_est))
    f0, logspc, f0_est, logspc_est = f0[:T], logspc[:T], f0_est[:T], logspc_est[:T]
    v = f0 > 0
    far = v.copy()
    for s in range(-3, 4):
        far &= np.roll(v, s)
    far[:3] = far[-3:] = False
    agree = float(np.mean(v == (f0_est > 0)))
    ferr = float(np.median(np.abs(f0_est[far] / f0[far] - 1.0)))
    fr = np.arange(257) * FS / 512
    band = (fr >= 100) & (fr <= 7000)
    d = logspc_est[far][:, band] - logspc[far][:, band]
    d = d - d.mean(axis=1, keepdims=True)
    rms = float(np.median(np.sqrt(np.mean(d * d, axis=1))))
    return ferr, agree, rms
