"""Restatement of v100_resample (include/v100.h): polyphase sinc resampling over a packed fp32 tap table, accumulated
in float64 with numpy.

For utterance b of length len[b], rates reduced by their gcd to o -> n and torchaudio's kernel half-width w:
    y[b, j n + p] = sum_i taps[off[p] + i] * x[b, j o + start[p] + i - w],   x = 0 outside [0, len[b]),
out_len[b] = out_length(len[b]) (ceil(n len[b] / o) up to torchaudio's float32 rounding) and samples
[out_len[b], L_out) are 0.  The table is the one
voice100_b200.data_modules.pack_resample_kernel builds from torchaudio's _get_sinc_resample_kernel; with the dense
kernel instead it is torchaudio's conv1d evaluated in float64 (_apply_sinc_resample_kernel).
"""
from __future__ import annotations

import numpy as np


def out_length(length: int, o: int, n: int) -> int:
    """torchaudio's output length: its conv1d yields n (length // o + 1) samples, sliced at
    torch.ceil(torch.as_tensor(n * length / o)) -- a float64 quotient rounded to float32, then ceil."""
    L = int(length)
    return min(int(np.ceil(np.float32(n * L / o))), n * (L // o + 1))


def resample_packed(x: np.ndarray, lengths, start, count, off, taps, o: int, n: int, w: int, L_out: int = None):
    """x [B, L] (float or int16 PCM, scaled by 1/32768), lengths [B] -> (y float64 [B, L_out], out_len int64 [B])."""
    x = np.asarray(x)
    xf = x.astype(np.float64) / 32768.0 if x.dtype == np.int16 else x.astype(np.float32).astype(np.float64)
    B, L = xf.shape
    if L_out is None:
        L_out = out_length(L, o, n)
    taps = np.asarray(taps, np.float32).astype(np.float64)
    y = np.zeros((B, L_out), np.float64)
    out_len = np.zeros(B, np.int64)
    for b in range(B):
        lb = min(max(int(lengths[b]), 0), L)
        ol = min(out_length(lb, o, n), L_out)
        out_len[b] = ol
        if ol == 0:
            continue
        K = 2 * w + o
        frames = (ol + n - 1) // n
        # zero-padded row: index m of xp is sample m - w
        xp = np.zeros(w + (frames - 1) * o + K + 1, np.float64)
        xp[w:w + lb] = xf[b, :lb]
        for p in range(n):
            c, s, f = int(count[p]), int(start[p]), int(off[p])
            js = np.arange(frames)
            if c == 0:
                acc = np.zeros(frames)
            else:
                idx = js[:, None] * o + s + np.arange(c)[None, :]       # xp index = sample + w
                acc = xp[idx] @ taps[f:f + c]
            q = js * n + p
            keep = q < ol
            y[b, q[keep]] = acc[keep]
    return y, out_len
