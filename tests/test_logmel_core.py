"""The FFT index math used by the CUDA log-mel kernel (csrc/logmel_core.h compiles for host and device):
built here with g++ and checked against numpy.fft.rfft, plus the full host restatement of one frame
against the oracle's mel pipeline."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

HARNESS = r"""
#include "logmel_core.h"
#include <cmath>
using namespace v100;
extern "C" void fft16_host(float* v) { fft16(reinterpret_cast<cpx*>(v)); }
// the 16-thread register decomposition of logmel.cu, thread by thread: two fft16 passes around the stride-17
// exchange, then the conjugate partner Z[256-k] taken from register 15-k2 of lane (16-q)&15 (own register (16-k2)&15
// for q = 0) -- what the kernel fetches with __shfl_sync -- and both bins of the pair from one complex multiply
extern "C" void rfft512_power_host(const float* frame, float* power) {
  static cpx tw[512];
  for (int k = 0; k < 512; ++k) { tw[k].x = (float)cos(-2.0*M_PI*k/512.0); tw[k].y = (float)sin(-2.0*M_PI*k/512.0); }
  cpx E[16 * 17], R[16][16];
  for (int q = 0; q < 16; ++q) {            // thread q: FFT over r, twiddle, write column q of the exchange
    cpx v[16];
    for (int r = 0; r < 16; ++r) { const int n = q + 16 * r; v[r] = cpx{frame[2 * n], frame[2 * n + 1]}; }
    fft16(v);
    for (int k1 = 0; k1 < 16; ++k1) E[k1 * 17 + q] = cmul(v[k1], tw[(2 * q * k1) & 511]);
  }
  for (int k1 = 0; k1 < 16; ++k1) {         // thread k1: FFT over q -> registers R[k1][k2] = Z[k1 + 16 k2]
    for (int q = 0; q < 16; ++q) R[k1][q] = E[k1 * 17 + q];
    fft16(R[k1]);
  }
  for (int q = 0; q < 16; ++q) {
    const int partner = (16 - q) & 15;
    for (int k2 = 0; k2 < 8; ++k2) {
      const cpx zn = q == 0 ? R[0][(16 - k2) & 15] : R[partner][15 - k2];
      const cpx w32 = cpx{(float)cos(-2.0*M_PI*k2/32.0), (float)sin(-2.0*M_PI*k2/32.0)};
      const int k = q + 16 * k2;
      rfft512_power_both(R[q][k2], zn, cmul(tw[q], w32), &power[k], &power[256 - k]);
    }
  }
  power[128] = rfft512_power_pair(R[0][8], R[0][8], cpx{0.0f, -1.0f});
}
"""


@pytest.fixture(scope="module")
def host_lib(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("logmel_core"))
    src = os.path.join(d, "h.cpp")
    with open(src, "w") as f:
        f.write(HARNESS)
    so = os.path.join(d, "h.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-I", os.path.join(ROOT, "voice100_b200", "csrc"), "-o", so, src])
    return ctypes.CDLL(so)


@pytest.fixture(scope="module")
def host_fft(host_lib):
    def run(frame):
        frame = np.ascontiguousarray(frame, np.float32)
        out = np.zeros(257, np.float32)
        host_lib.rfft512_power_host(frame.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p))
        return out
    return run


def test_rfft512_power_matches_numpy(host_fft):
    rng = np.random.default_rng(0)
    for trial in range(4):
        x = rng.standard_normal(512).astype(np.float32) * (10.0 ** (trial - 2))
        ref = np.abs(np.fft.rfft(x.astype(np.float64))) ** 2
        got = host_fft(x)
        assert np.max(np.abs(got - ref)) <= 3e-6 * ref.max()
    imp = np.zeros(512, np.float32)
    imp[3] = 1.0
    np.testing.assert_allclose(host_fft(imp), np.ones(257), rtol=1e-5)            # flat spectrum
    tone = np.cos(2 * np.pi * 37 * np.arange(512) / 512).astype(np.float32)
    p = host_fft(tone)
    assert p.argmax() == 37 and abs(p[37] - 256.0 ** 2) < 1e-2 * 256.0 ** 2       # one bin, N/2 amplitude


def test_fft16_matches_numpy(host_lib):
    rng = np.random.default_rng(1)
    for _ in range(5):
        v = (rng.standard_normal(16) + 1j * rng.standard_normal(16)).astype(np.complex64)
        buf = v.view(np.float32).copy()
        host_lib.fft16_host(buf.ctypes.data_as(ctypes.c_void_p))
        np.testing.assert_allclose(buf.view(np.complex64), np.fft.fft(v.astype(np.complex128)), atol=2e-6 * 16)


def test_shared_memory_accesses_are_conflict_free():
    """Bank arithmetic of logmel.cu.  64-bit exchange accesses of one half-warp (16 lanes x 8 bytes = one 128-byte
    wavefront when the lanes hit 16 different bank pairs): writes E[k1*17 + q], reads E[q*17 + qq].  32-bit power
    stores of a whole warp into P[bin*33 + frame] (the two half-warps hold frames 16 apart): 32 distinct banks for
    both the k = q + 16 k2 and the 256 - k stores.  Mel-phase loads P[(s0+tap)*33 + lane]: 32 distinct banks."""
    def bank_pairs(idx):
        return len({i % 16 for i in idx})
    for k1 in range(16):
        assert bank_pairs([k1 * 17 + q for q in range(16)]) == 16
    for qq in range(16):
        assert bank_pairs([q * 17 + qq for q in range(16)]) == 16      # what the padding to 17 buys
        assert bank_pairs([q * 16 + qq for q in range(16)]) == 1       # ... and what 16 would cost
    for fl in range(16):
        for k2 in range(8):
            lo = [(q + 16 * k2) * 33 + fl + 16 * h for h in range(2) for q in range(16)]
            hi = [(256 - q - 16 * k2) * 33 + fl + 16 * h for h in range(2) for q in range(16)]
            assert len({i % 32 for i in lo}) == 32 and len({i % 32 for i in hi}) == 32
            bad = [(q + 16 * k2) * 33 + fl + h for h in range(2) for q in range(16)]   # adjacent frames would collide
            assert len({i % 32 for i in bad}) < 32
    for row in (0, 7, 256):
        assert len({(row * 33 + lane) % 32 for lane in range(32)}) == 32


def test_every_power_bin_is_written_once():
    """The pair scheme of logmel.cu covers bins 0..256 exactly once: k = q + 16 k2 (k2 < 8), its partner 256 - k,
    and bin 128 from lane 0."""
    seen = [0] * 257
    for q in range(16):
        for k2 in range(8):
            k = q + 16 * k2
            seen[k] += 1
            seen[256 - k] += 1
    seen[128] += 1
    assert seen == [1] * 257


def test_frame_pipeline_matches_oracle(host_fft):
    import torch
    import v100_oracle as orc
    from voice100_b200 import synth
    from voice100_b200.data_modules import mel_filterbank, sparse_filterbank
    w = synth.harmonic_waveform(1, 4000, seed=3)[0]
    L = len(w)
    start, count, off, fw = sparse_filterbank(mel_filterbank(16000, 512, 64))
    win = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(400) / 400)
    ref = orc.logmel_clip(torch.from_numpy(w)).numpy()
    for t in (0, 1, 7, L // 160):                                  # first frames reflect left, last reflects right
        frame = np.zeros(512, np.float32)
        for m in range(56, 456):
            i = 160 * t - 256 + m
            i = -i if i < 0 else i
            i = 2 * (L - 1) - i if i >= L else i
            frame[m] = w[i] * win[m - 56]
        p = host_fft(frame)
        mel = np.array([np.dot(fw[off[m]:off[m] + count[m]], p[start[m]:start[m] + count[m]]) for m in range(64)])
        np.testing.assert_allclose(np.log(mel + 1e-6), ref[t], rtol=0, atol=2e-3)
