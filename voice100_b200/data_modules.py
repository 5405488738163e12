"""Log-mel front end with the reference's interface (voice100/data_modules.py:23-26,262-292).

`MelSpectrogramAudioTransform` keeps the reference's constructor arguments, `audio_size` property and
`.melspec(waveform[..., L]) -> [..., n_mels, 1 + L//hop]` call; the arithmetic is one fused CUDA kernel
(v100_logmel) instead of torchaudio's reflect-pad + cuFFT + sgemm chain.  `logmel_batch` is the batched
form of what `EncodedCacheDataset` + `generate_audio_text_batch` (data_modules.py:210-234,446-455) build
per utterance on the CPU: per-clip features padded with BLANK_AUDIO.

`resample` is torchaudio.functional.resample on the device (v100_resample), the step the reference's `forward`
takes between load and the mel spectrogram when a file is not at 16 kHz (data_modules.py:288-289);
`logmel_batch(orig_freq=...)` and `forward(orig_freq=...)` apply it first.
"""
from __future__ import annotations

import math
import warnings
from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np
import torch
from torch import nn

from . import kernels as K
from ._lib import V100Error

MELSPEC_DIM = 64
LOG_OFFSET = 1e-6
BLANK_AUDIO = math.log(LOG_OFFSET)


def _hz_to_mel_htk(f: float) -> float:
    return 2595.0 * math.log10(1.0 + f / 700.0)


def mel_filterbank(sample_rate: int, n_fft: int, n_mels: int) -> np.ndarray:
    """HTK triangular filters, norm=None, f_min=0, f_max=sr/2 -> fb[n_fft//2+1, n_mels] fp32.  A host-side
    constant table; built with the same fp32 torch ops, in the same order, as
    torchaudio.functional.melscale_fbanks so the weights are bit-identical to the reference's."""
    n_freqs = n_fft // 2 + 1
    all_freqs = torch.linspace(0, sample_rate // 2, n_freqs)
    m_pts = torch.linspace(_hz_to_mel_htk(0.0), _hz_to_mel_htk(float(sample_rate // 2)), n_mels + 2)
    f_pts = 700.0 * (10.0 ** (m_pts / 2595.0) - 1.0)
    f_diff = f_pts[1:] - f_pts[:-1]
    slopes = f_pts.unsqueeze(0) - all_freqs.unsqueeze(1)
    down = (-1.0 * slopes[:, :-2]) / f_diff[:-1]
    up = slopes[:, 2:] / f_diff[1:]
    return torch.max(torch.zeros(1), torch.min(down, up)).numpy()


def sparse_filterbank(fb: np.ndarray):
    """Column-compressed form consumed by v100_logmel: per filter (first bin, count, offset) + weights."""
    start, count, off, w = [], [], [], []
    for m in range(fb.shape[1]):
        nz = np.nonzero(fb[:, m])[0]
        s, e = (int(nz[0]), int(nz[-1]) + 1) if len(nz) else (0, 0)
        start.append(s); count.append(e - s); off.append(len(w))
        w.extend(fb[s:e, m].tolist())
    return (np.asarray(start, np.int32), np.asarray(count, np.int32), np.asarray(off, np.int32),
            np.asarray(w, np.float32))


# ------------------------------------------------------------------------------------------------ resampling

_HANN, _KAISER = "sinc_interp_hann", "sinc_interp_kaiser"
_KAISER_BETA = 14.769656459379492            # torchaudio's default beta for sinc_interp_kaiser


def _check_rates(orig_freq, new_freq):
    if orig_freq <= 0.0 or new_freq <= 0.0:
        raise ValueError("Original frequency and desired frequecy should be positive")


def sinc_resample_kernel(orig_freq: int, new_freq: int, gcd: int, lowpass_filter_width: int = 6,
                         rolloff: float = 0.99, resampling_method: str = _HANN, beta: Optional[float] = None):
    """torchaudio.functional's `_get_sinc_resample_kernel` rebuilt with the same float64 torch ops in the same order,
    so the fp32 taps are bit-identical to it for both windows; it raises what torchaudio raises for non-integer rates,
    an unknown method or lowpass_filter_width <= 0.
    -> (kernel fp32 [n, 1, 2 width + o], width, inside bool [n, 2 width + o]), o = orig_freq // gcd, n = new_freq // gcd.
    `inside` marks the taps whose sinc argument t lies strictly within +-lowpass_filter_width, before torchaudio clamps
    it there: per phase a contiguous run, since t grows with the column."""
    if not (int(orig_freq) == orig_freq and int(new_freq) == new_freq):
        raise Exception("Frequencies must be of integer type to ensure quality resampling computation. "
                        "To work around this, manually convert both frequencies to integer values "
                        "that maintain their resampling rate ratio before passing them into the function.")
    if resampling_method in ("sinc_interpolation", "kaiser_window"):
        method_map = {"sinc_interpolation": _HANN, "kaiser_window": _KAISER}
        warnings.warn(f'"{resampling_method}" resampling method name is being deprecated and replaced by '
                      f'"{method_map[resampling_method]}" in the next release. The default behavior remains unchanged.',
                      stacklevel=3)
        resampling_method = method_map[resampling_method]
    elif resampling_method not in (_HANN, _KAISER):
        raise ValueError("Invalid resampling method: {}".format(resampling_method))
    orig_freq = int(orig_freq) // gcd
    new_freq = int(new_freq) // gcd
    if lowpass_filter_width <= 0:
        raise ValueError("Low pass filter width should be positive.")
    base_freq = min(orig_freq, new_freq)
    base_freq *= rolloff
    width = math.ceil(lowpass_filter_width * orig_freq / base_freq)
    idx = torch.arange(-width, width + orig_freq, dtype=torch.float64)[None, None] / orig_freq
    t = torch.arange(0, -new_freq, -1)[:, None, None] / new_freq + idx
    t *= base_freq
    inside = (t.abs() < lowpass_filter_width)[:, 0]
    t = t.clamp_(-lowpass_filter_width, lowpass_filter_width)
    if resampling_method == _HANN:
        window = torch.cos(t * math.pi / lowpass_filter_width / 2) ** 2
    else:
        if beta is None:
            beta = _KAISER_BETA
        beta_tensor = torch.tensor(float(beta))
        window = torch.i0(beta_tensor * torch.sqrt(1 - (t / lowpass_filter_width) ** 2)) / torch.i0(beta_tensor)
    t *= math.pi
    scale = base_freq / orig_freq
    kernels = torch.where(t == 0, torch.tensor(1.0).to(t), t.sin() / t)
    kernels *= window * scale
    return kernels.to(dtype=torch.float32), width, inside


def pack_resample_kernel(kernel: torch.Tensor, inside: torch.Tensor):
    """Per phase, the run of taps with |t| < lowpass_filter_width -> (start, count, off) int32 [n] and taps fp32, the
    table v100_resample reads (phase p's run covers dense columns [start[p], start[p] + count[p]) and is
    taps[off[p] ...]).  The taps it drops are the ones where torchaudio clamps t to +-lowpass_filter_width:
      - sinc_interp_hann: the window there is cos(pi / 2)^2 ~ 4e-33 and the product rounds to exactly 0 in fp32, so the
        run is exactly the non-zero taps;
      - sinc_interp_kaiser: every dropped tap has the single value scale * sin(pi w) / (pi w) / I0(beta) (w =
        lowpass_filter_width), which float64 sin(pi w) makes at most 1.3e-16 * scale / I0(beta) in magnitude: below
        1e-21 for the default beta (I0(14.77) = 2.6e5), below 1.3e-16 for any beta >= 0.
    torchaudio multiplies those taps with real samples, so a Kaiser result may differ from it by that much per tap."""
    k = kernel[:, 0].numpy()
    ins = inside.numpy()
    start, count, off, taps = [], [], [], []
    for p in range(k.shape[0]):
        nz = np.nonzero(ins[p])[0]
        s, e = (int(nz[0]), int(nz[-1]) + 1) if len(nz) else (0, 0)
        start.append(s); count.append(e - s); off.append(len(taps))
        taps.extend(k[p, s:e].tolist())
    return (np.asarray(start, np.int32), np.asarray(count, np.int32), np.asarray(off, np.int32),
            np.asarray(taps, np.float32))


@dataclass
class ResampleTable:
    """The packed polyphase table of one (rates, parameters) on one device."""
    o: int
    n: int
    width: int
    start: torch.Tensor
    count: torch.Tensor
    off: torch.Tensor
    taps: torch.Tensor


_resample_tables = {}


def resample_table(orig_freq, new_freq, lowpass_filter_width=6, rolloff=0.99, resampling_method=_HANN, beta=None,
                   device="cuda") -> ResampleTable:
    """The device table for these parameters, built on the host once per (rates, parameters, device) and cached.
    Building uploads it, so it must happen outside CUDA-graph capture: a captured call whose table is not cached yet
    raises (run the call once before capturing)."""
    _check_rates(orig_freq, new_freq)
    gcd = math.gcd(int(orig_freq), int(new_freq))
    dev = torch.device(device)
    if dev.type == "cuda" and dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    key = (orig_freq / gcd, new_freq / gcd, lowpass_filter_width, float(rolloff), resampling_method,
           None if beta is None else float(beta), str(dev))
    tab = _resample_tables.get(key)
    if tab is None:
        kernel, width, inside = sinc_resample_kernel(orig_freq, new_freq, gcd, lowpass_filter_width, rolloff,
                                                     resampling_method, beta)
        if dev.type == "cuda" and torch.cuda.is_current_stream_capturing():
            raise V100Error("the resampling table for these rates is not built yet: run the call once before graph "
                            "capture so that the table is built there")
        arrs = [torch.from_numpy(a).to(dev) for a in pack_resample_kernel(kernel, inside)]
        tab = ResampleTable(int(orig_freq) // gcd, int(new_freq) // gcd, width, *arrs)
        _resample_tables[key] = tab
    return tab


def resampled_length(length, orig_freq: int, new_freq: int):
    """The number of samples torchaudio.functional.resample returns for `length` input samples (rates reduced by their
    gcd to o -> n): its conv1d gives n (length // o + 1) samples and it keeps the first
    torch.ceil(torch.as_tensor(n * length / o)), a float64 quotient rounded to a float32 tensor.  That is
    ceil(n length / o) while float32 resolves 1/o at n length / o (below 2^15 output samples at 44.1 kHz, 2^22 at
    48 kHz); past that it can be one sample shorter (or, beyond 2^25, longer) than the exact ceiling, and v100_resample
    computes the same rounding.  `length` an int or an integer tensor."""
    g = math.gcd(int(orig_freq), int(new_freq))
    o, n = int(orig_freq) // g, int(new_freq) // g
    if isinstance(length, torch.Tensor):
        L = length.to(torch.int64)
        return torch.minimum(torch.ceil((L.double() * n / o).float()).long(), n * (torch.div(L, o, rounding_mode="floor") + 1))
    L = int(length)
    return min(int(math.ceil(float(np.float32(n * L / o)))), n * (L // o + 1))


def resample(waveform: torch.Tensor, orig_freq: int, new_freq: int, lowpass_filter_width: int = 6,
             rolloff: float = 0.99, resampling_method: str = _HANN, beta: Optional[float] = None,
             lengths: Optional[torch.Tensor] = None):
    """torchaudio.functional.resample on the device (v100_resample): same signature, same taps, same output length,
    and the same exceptions for non-positive or non-integer rates, lowpass_filter_width <= 0 and an unknown method.
    waveform fp32 or int16 PCM (scaled by 1/32768) on a CUDA device; anything else raises V100Error.
      - without `lengths`: [..., L] -> fp32 [..., L_out(L)];
      - with `lengths` (int [B], on the device for no host synchronisation): [B, L_max] (any row pitch) ->
        (out fp32 [B, L_out(L_max)], out_len int32 [B] = L_out(lengths)); row b is what torchaudio returns for
        waveform[b, :lengths[b]], followed by zeros.
    L_out(L) is torchaudio's output length, `resampled_length`: ceil(n L / o) up to a float32 rounding torchaudio
    applies for long clips.
    orig_freq == new_freq returns the waveform unchanged (as fp32), as torchaudio does.  The result is accumulated in
    fp32 by the kernel, one fixed-order chain per sample; torchaudio's conv1d rounds differently in the last bits."""
    _check_rates(orig_freq, new_freq)
    if not waveform.is_cuda:
        raise V100Error("resample runs only on CUDA tensors (no CPU path)")
    if waveform.dtype not in (torch.float32, torch.int16):
        raise V100Error(f"resample: waveforms must be float32 or int16 PCM, got {waveform.dtype}")
    if lengths is not None and (waveform.dim() != 2 or tuple(lengths.shape) != (waveform.shape[0],)):
        raise V100Error(f"resample: with lengths the waveform must be [B, L] and lengths [B]; got "
                        f"{tuple(waveform.shape)} and {tuple(lengths.shape)}")
    if lengths is not None and (lengths.dtype.is_floating_point or lengths.dtype == torch.bool):
        raise V100Error(f"resample: lengths must be an integer tensor, got {lengths.dtype}")
    if orig_freq == new_freq:
        out = waveform.float() / 32768.0 if waveform.dtype == torch.int16 else waveform
        return out if lengths is None else (out, lengths.to(device=waveform.device, dtype=torch.int32))
    tab = resample_table(orig_freq, new_freq, lowpass_filter_width, rolloff, resampling_method, beta,
                         waveform.device)
    lead, L = waveform.shape[:-1], waveform.shape[-1]
    wav = waveform if lengths is not None else waveform.reshape(-1, L)
    if wav.stride(-1) != 1 or (wav.shape[0] > 1 and wav.stride(0) < L):
        wav = wav.contiguous()
    if lengths is None:
        lens = torch.full((wav.shape[0],), L, dtype=torch.int32, device=wav.device)
    else:
        lens = lengths.to(device=wav.device, dtype=torch.int32).contiguous()
    out, out_len = K.resample(wav, lens, tab, resampled_length(L, orig_freq, new_freq))
    return out.reshape(*lead, out.shape[-1]) if lengths is None else (out, out_len)


class MelSpectrogramAudioTransform(nn.Module):
    def __init__(self, sample_rate: int = 16000, n_fft: int = 512, win_length: int = 400, hop_length: int = 160,
                 n_mels: int = MELSPEC_DIM, log_offset: float = LOG_OFFSET) -> None:
        super().__init__()
        # (512, 400, 160, 64) -- the only configuration the reference ever builds, data_modules.py:266-269 -- runs the tuned
        # kernel; any other one the generic kernel (v100_logmel_generic)
        if n_fft < 8 or n_fft > 2048 or (n_fft & (n_fft - 1)) != 0:
            raise V100Error(f"n_fft={n_fft}: powers of two in [8, 2048] are supported")
        if not (0 < win_length <= n_fft) or hop_length <= 0 or n_mels <= 0:
            raise V100Error("need 0 < win_length <= n_fft, hop_length > 0, n_mels > 0")
        self.sample_rate, self.n_fft, self.win_length, self.hop_length = sample_rate, n_fft, win_length, hop_length
        self.n_mels, self.log_offset = n_mels, log_offset
        fb = mel_filterbank(sample_rate, n_fft, n_mels)
        for name, arr in zip(("fb_start", "fb_count", "fb_off", "fb_w"), sparse_filterbank(fb)):
            self.register_buffer(name, torch.from_numpy(arr), persistent=False)

    @property
    def audio_size(self) -> int:
        return self.n_mels

    @property
    def _config(self):
        return (self.n_fft, self.win_length, self.hop_length, self.n_mels)

    def _fb(self, device):
        if self.fb_w.device != device:
            self.to(device)
        return (self.fb_start, self.fb_count, self.fb_off, self.fb_w)

    def num_frames(self, num_samples):
        return 1 + num_samples // self.hop_length

    def melspec(self, waveform: torch.Tensor) -> torch.Tensor:
        """Mel power spectrogram, `[..., L] -> [..., 64, 1 + L//160]` fp32 (what the reference's
        `self.melspec` torchaudio module returns, data_modules.py:290)."""
        if not waveform.is_cuda:
            raise V100Error("MelSpectrogramAudioTransform runs only on CUDA tensors (no CPU path)")
        lead, L = waveform.shape[:-1], waveform.shape[-1]
        if L <= self.n_fft // 2:
            raise V100Error(f"clips must be longer than {self.n_fft // 2} samples (reflect padding)")
        wav = self._samples(waveform.reshape(-1, L))
        lengths = torch.full((wav.shape[0],), L, dtype=torch.int32, device=wav.device)
        T = self.num_frames(L)
        out, _ = K.logmel(wav, lengths, self._fb(wav.device), self.log_offset, T, K.MEL_POWER_F32_NCW, self._config)
        return out.valid().reshape(*lead, self.n_mels, T)

    @staticmethod
    def _samples(waveform: torch.Tensor) -> torch.Tensor:
        """fp32 samples, or int16 PCM passed through untouched (the kernel scales by 1/32768, which is what
        torchaudio.load returns for a 16-bit WAV -- data_modules.py:288 -- so both forms give identical features)."""
        if waveform.dtype == torch.int16:
            return waveform.contiguous()
        return waveform.to(torch.float32).contiguous()

    def logmel_batch(self, waveform: torch.Tensor, lengths: torch.Tensor, ncw_bf16: bool = False, ncw_dtype=None,
                     orig_freq: Optional[int] = None):
        """waveform fp32 (or int16 PCM) [B, L_max], lengths [B] samples ->
        (audio fp32 [B, T_max, 64] padded with BLANK_AUDIO  |  16-bit Ncw [B, 64, pitch] when `ncw_dtype`
         (torch.bfloat16 / torch.float16) or `ncw_bf16` is given,  audio_len int32 [B] = 1 + len // 160).
        Host-resident `lengths` are validated like torchaudio does (reflect padding needs > n_fft/2 samples, 0 =
        an empty filler slot); device-resident ones are clamped to [0, L_max] by the kernel.
        `orig_freq`, the rate of the waveform when it is not `sample_rate`: the batch is resampled first (`resample`
        with lengths: one more kernel, no host synchronisation), and host lengths are validated after resampling."""
        if ncw_bf16 and ncw_dtype is None:
            ncw_dtype = torch.bfloat16
        if not waveform.is_cuda:
            raise V100Error("MelSpectrogramAudioTransform runs only on CUDA tensors (no CPU path)")
        if orig_freq is not None and orig_freq != self.sample_rate:
            if not lengths.is_cuda and lengths.numel():
                if int(lengths.max()) > waveform.shape[1] or int(lengths.min()) < 0:
                    raise V100Error(f"clip lengths must be in [0, {waveform.shape[1]}]; got [{int(lengths.min())}, "
                                    f"{int(lengths.max())}]")
                self._check_lengths(resampled_length(lengths, orig_freq, self.sample_rate),
                                    resampled_length(waveform.shape[1], orig_freq, self.sample_rate))
            waveform, lengths = resample(waveform, orig_freq, self.sample_rate, lengths=lengths)
        wav = self._samples(waveform)
        if not lengths.is_cuda and lengths.numel():
            self._check_lengths(lengths, wav.shape[1])
        lengths = lengths.to(device=wav.device, dtype=torch.int32).contiguous()
        T = self.num_frames(wav.shape[1])
        mode = K.MEL_LOG_F32_NTC if ncw_dtype is None else (K.MEL_LOG_F16_NCW if K.dt(ncw_dtype) == 1 else K.MEL_LOG_BF16_NCW)
        return K.logmel(wav, lengths, self._fb(wav.device), self.log_offset, T, mode, self._config)

    def _check_lengths(self, lengths: torch.Tensor, L: int):
        lo, hi = int(lengths.min()), int(lengths.max())
        if hi > L or ((lengths > 0) & (lengths <= self.n_fft // 2)).any():
            raise V100Error(f"clip lengths must be 0 (empty slot) or in ({self.n_fft // 2}, {L}]; got [{lo}, {hi}]")

    def forward(self, waveform: torch.Tensor, orig_freq: Optional[int] = None) -> torch.Tensor:
        """One clip `[L] -> [T, 64]` log-mel features.  The reference's forward takes a file path, loads it and
        resamples to `sample_rate` when the file's rate differs (data_modules.py:287-289); file I/O is outside the
        accelerated path, and `orig_freq` (the clip's rate) does the resampling on the device."""
        if orig_freq is not None and orig_freq != self.sample_rate:
            if not waveform.is_cuda:
                raise V100Error("MelSpectrogramAudioTransform runs only on CUDA tensors (no CPU path)")
            waveform = resample(waveform, orig_freq, self.sample_rate)
        return torch.log(self.melspec(waveform).transpose(-1, -2) + self.log_offset)
