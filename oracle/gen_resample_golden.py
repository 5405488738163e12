"""Generate tests/golden/resample.npz from torchaudio (no reference checkout needed).

    python oracle/gen_resample_golden.py

Stores, for a handful of rate pairs and parameters, torchaudio's dense fp32 kernel packed into the per-phase runs
v100_resample reads, torchaudio.functional.resample of seeded inputs at a few lengths, and the log-mel features
(oracle v100_oracle.logmel_clip) of one 44.1 kHz clip resampled to 16 kHz by torchaudio, which is what the reference's
MelSpectrogramAudioTransform.forward computes for a 44.1 kHz file (voice100/data_modules.py:287-292).
"""
import math
import os
import sys

import numpy as np
import torch
import torchaudio.functional as AF
from torchaudio.functional.functional import _get_sinc_resample_kernel

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [ROOT, HERE]

import v100_oracle as orc  # noqa: E402
from voice100_b200.data_modules import pack_resample_kernel, sinc_resample_kernel  # noqa: E402

RATIOS = [(48000, 16000), (44100, 16000), (32000, 16000), (24000, 16000), (22050, 16000), (11025, 16000),
          (8000, 16000), (16000, 22050), (16000, 24000), (16000, 44100), (16000, 48000)]
TABLES = ([(a, b, 6, 0.99, m) for a, b in RATIOS for m in ("sinc_interp_hann", "sinc_interp_kaiser")]
          + [(44100, 16000, 16, 0.945, "sinc_interp_hann"), (16000, 48000, 16, 0.945, "sinc_interp_kaiser")])
OUTPUTS = [(44100, 16000), (48000, 16000), (22050, 16000), (8000, 16000), (16000, 48000), (16000, 44100)]
LENGTHS = [1, 37, 1000, 2003]


def tag(a, b, lpw=6, rolloff=0.99, method="sinc_interp_hann"):
    return f"{a}_{b}_{lpw}_{rolloff}_{method.split('_')[-1]}"


def main():
    out = {}
    for a, b, lpw, ro, m in TABLES:
        g = math.gcd(a, b)
        ref, width = _get_sinc_resample_kernel(a, b, g, lpw, ro, m, None)
        kernel, w2, inside = sinc_resample_kernel(a, b, g, lpw, ro, m, None)
        assert w2 == width and torch.equal(kernel, ref)
        t = tag(a, b, lpw, ro, m)
        for name, arr in zip(("start", "count", "off", "taps"), pack_resample_kernel(kernel, inside)):
            out[f"table/{t}/{name}"] = arr
        out[f"table/{t}/width"] = np.int64(width)
    rng = np.random.default_rng(20261020)
    for a, b in OUTPUTS:
        for L in LENGTHS:
            x = (0.3 * rng.standard_normal(L)).astype(np.float32)
            out[f"x/{a}_{b}/{L}"] = x
            out[f"y/{a}_{b}/{L}"] = AF.resample(torch.from_numpy(x), a, b).numpy()
    # one 44.1 kHz clip (0.5 s of a chirp plus noise, 16-bit PCM as a WAV file holds it) -> torchaudio.load's scaling
    # -> torchaudio resample -> log-mel
    n = 22050
    t = np.arange(n) / 44100.0
    wave = 0.4 * np.sin(2 * np.pi * (200 * t + 1800 * t * t)) + 0.05 * rng.standard_normal(n)
    clip = np.round(wave * 32767).astype(np.int16)
    clip16 = AF.resample(torch.from_numpy(clip.astype(np.float32) / 32768.0), 44100, 16000)
    out["clip44k"] = clip
    out["clip44k_resampled"] = clip16.numpy()
    out["clip44k_logmel"] = orc.logmel_clip(clip16).numpy()
    path = os.path.join(ROOT, "tests", "golden", "resample.npz")
    np.savez_compressed(path, **out)
    print(f"wrote {path}: {len(out)} arrays, {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
