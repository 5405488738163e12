"""Mel-cepstrum -> log-spectrum on the inference path (SURVEY.md section 8f #4), and the WORLD vocoder.

The reference's shipped TTS config trains AlignTextToAudio on 25 mel-cepstral coefficients (config/tts_en_base.yaml:29
`vocoder: world_mcep`) and converts them back with a fixed matrix after `predict`
(voice100/export_onnx.py:81-97 `AlignTextToAudioPredict`, voice100/vocoder.py:115-123 `create_mc2sp_matrix`).
Un-normalisation and that matrix are both linear, so here they are folded into the projection layer: the head GEMM
emits the 257 log-spectrum bins directly and the conversion costs nothing at run time.
WORLD waveform synthesis (the reference's WORLDVocoder.decode, pyworld on the host) runs on the device through
`WORLDVocoder` (v100_world_synthesize); WORLD analysis (encode) is not on the inference path and stays out of scope.
"""
from __future__ import annotations

from typing import Tuple

import numpy as np
import torch
from torch import nn

from . import kernels as K
from ._lib import V100Error
from .blocks import PreparedCache, require_eval_cuda
from .v2 import AlignTextToAudio, _run_lstm


def _warp_operator(n_in: int, n_out: int, alpha: float) -> np.ndarray:
    """Matrix A [n_in, n_out] of the all-pass frequency transformation (SPTK freqt): warped = cepstrum @ A.
    Built by pushing the coefficients through the recursion one at a time, last coefficient first; the state is
    kept for all unit inputs at once (one row per input coefficient)."""
    state = np.zeros((n_in, n_out))
    b = 1.0 - alpha * alpha
    for i in range(n_in - 1, -1, -1):
        nxt = np.empty_like(state)
        nxt[:, 0] = alpha * state[:, 0]
        nxt[i, 0] += 1.0                                   # unit cepstrum i contributes its coefficient i now
        if n_out > 1:
            nxt[:, 1] = b * state[:, 0] + alpha * state[:, 1]
        for j in range(2, n_out):
            nxt[:, j] = state[:, j - 1] + alpha * (state[:, j] - nxt[:, j - 1])
        state = nxt
    return state


def create_mc2sp_matrix(fftlen: int, order: int, alpha: float) -> np.ndarray:
    """float64 [order+1, fftlen//2+1]: logspc = mcep @ M, PySPTK `mc2sp` conventions (vocoder.py:115-123)."""
    c = _warp_operator(order + 1, fftlen // 2 + 1, -alpha)
    c[:, 0] *= 2.0
    even = np.concatenate([c, c[:, :0:-1]], axis=1)
    return np.fft.rfft(even, axis=1).real


class AlignTextToAudioPredict(nn.Module):
    """`predict` followed by the mel-cepstrum -> log-spectrum matrix (export_onnx.py:81-97), as one fused head.
    forward(aligntext, aligntext_len) -> (f0 [B,T'], logspc [B,T',257], codeap [B,T',A])."""

    def __init__(self, model: AlignTextToAudio, fftlen: int = 512, order: int = 24, alpha: float = 0.410) -> None:
        super().__init__()
        self.model = model
        if model.logspc_size == order + 1:
            self.register_buffer("mc2sp_matrix", torch.from_numpy(create_mc2sp_matrix(fftlen, order, alpha)).float())
        elif model.logspc_size == fftlen // 2 + 1:
            self.mc2sp_matrix = None
        else:
            raise V100Error(f"logspc_size {model.logspc_size} is neither {order + 1} mel-cepstra nor {fftlen // 2 + 1} bins")
        self._prepared = PreparedCache(self, self._prepare)
        self.eval()

    def _prepare(self):
        """Head producing [hasf0, f0, logspc(257), hascodeap, codeap] with un-normalisation (and mc2sp) folded in:
        rows of W' x + b' where x is the decoder output."""
        m, n = self.model, self.model.norm
        W, b = m.projection.weight.detach().double(), m.projection.bias.detach().double()
        S, A = m.logspc_size, m.codeap_size
        i_f0, i_sp, i_hc, i_ap = 1, 2, 2 + S, 2 + S + A
        rows_w = [W[0:1], n.f0_std.double()[:, None] * W[i_f0:i_f0 + 1]]
        rows_b = [b[0:1], n.f0_std.double() * b[i_f0:i_f0 + 1] + n.f0_mean.double()]
        Wsp = n.logspc_std.double()[:, None] * W[i_sp:i_sp + S]
        bsp = n.logspc_std.double() * b[i_sp:i_sp + S] + n.logspc_mean.double()
        if self.mc2sp_matrix is not None:
            M = self.mc2sp_matrix.double()
            Wsp, bsp = M.T @ Wsp, bsp @ M
        rows_w += [Wsp, W[i_hc:i_hc + A], n.codeap_std.double()[:, None] * W[i_ap:i_ap + A]]
        rows_b += [bsp, b[i_hc:i_hc + A], n.codeap_std.double() * b[i_ap:i_ap + A] + n.codeap_mean.double()]
        dtype = m.storage_dtype
        n_out = 1 + Wsp.shape[0] + A                       # un-normalisation is already in W', b': identity statistics
        dev = W.device
        return dict(w=torch.cat(rows_w, 0).to(dtype).contiguous(), b=torch.cat(rows_b, 0).float().contiguous(),
                    bins=Wsp.shape[0], ident=(torch.zeros(n_out, device=dev), torch.ones(n_out, device=dev)))

    def forward(self, aligntext: torch.Tensor, aligntext_len: torch.Tensor, t_max: int = None) -> Tuple[torch.Tensor, ...]:
        """`t_max`: decode the first t_max frames without reading the lengths back (default max(aligntext_len))."""
        m = self.model
        require_eval_cuda(self, aligntext)
        w, mw = self._prepared.get(), m._prepared.get()
        if t_max is None:
            t_max = int(aligntext_len.max())
        tm = K.ncw_to_tm(K.embedding_ncw(aligntext[:, :t_max].contiguous(), mw["table"]))
        tm = _run_lstm(tm, mw["lstm"], aligntext_len)
        x = m.decoder.run(K.tm_to_ncw(tm))
        # split + the f0 / codeap presence gates in one kernel (the statistics passed are the identity)
        _, f0, logspc, _, codeap = K.world_finalize(K.conv1x1_f32(x, w["w"], w["b"]), w["ident"][0], w["ident"][1],
                                                    True, w["bins"], m.codeap_size, 2)
        return f0, logspc, codeap


class WORLDVocoder:
    """WORLD synthesis on the device, in place of the reference's WORLDVocoder.decode (voice100/vocoder.py:89-102:
    pyworld.decode_aperiodicity + pyworld.synthesize, one utterance on a CPU core).  Only the configuration every model
    here emits is implemented: 16 kHz, 10 ms frames, 512-point FFT (257 log-spectrum bins, one coded-aperiodicity band).
    The algorithm is the restatement in oracle/world.py; parity with pyworld itself is unverified (DESIGN.md 3.8).
    Inputs are used as fp32, the precision the models produce them in."""

    def __init__(self, sample_rate: int = 16000, frame_period: float = 10.0, n_fft: int = 512) -> None:
        if (sample_rate, float(frame_period), n_fft) != (K.WORLD_FS, 10.0, K.WORLD_FFT):
            raise V100Error(f"WORLDVocoder: only sample_rate=16000, frame_period=10.0, n_fft=512 is implemented "
                            f"(got {sample_rate}, {frame_period}, {n_fft})")
        self.sample_rate, self.frame_period, self.n_fft = sample_rate, float(frame_period), n_fft

    def decode_batch(self, f0: torch.Tensor, logspc: torch.Tensor, codeap: torch.Tensor, frame_len: torch.Tensor = None,
                     max_samples: int = None):
        """Device tensors f0 [B, T], logspc [B, T, 257], codeap [B, T, 1] (fp32, any strides), frame_len int32 [B] or
        None -> (wav fp32 [B, Y], wav_len int32 [B], status int32 [B]); see kernels.world_synthesize.  No host sync."""
        if frame_len is not None:
            frame_len = frame_len.to(device=f0.device, dtype=torch.int32).contiguous()
        return K.world_synthesize(f0, logspc, codeap, frame_len, max_samples)

    def decode(self, f0, logspc, codeap, device=None) -> np.ndarray:
        """One utterance, like the reference: f0 [T], logspc [T, 257], codeap [T, 1] (numpy arrays or tensors)
        -> float64 numpy waveform [160 T].  Runs on `device` (default: the tensors' CUDA device, else the current one).
        Raises ValueError where WORLD has no defined behaviour (fewer than two frames, NaN or inf)."""
        if device is None:
            device = f0.device if isinstance(f0, torch.Tensor) and f0.is_cuda else torch.device(
                "cuda", torch.cuda.current_device())
        as_t = lambda x: torch.as_tensor(np.asarray(x.detach().cpu() if isinstance(x, torch.Tensor) else x),
                                         dtype=torch.float32).to(device)
        f0_t, sp_t, ap_t = as_t(f0).reshape(1, -1), as_t(logspc), as_t(codeap)
        T = f0_t.shape[1]
        sp_t = sp_t.reshape(1, T, -1)
        ap_t = ap_t.reshape(1, T, -1)
        wav, wav_len, status = self.decode_batch(f0_t, sp_t, ap_t)
        st = int(status[0])
        if st == K.WORLD_SHORT:
            raise ValueError("WORLD synthesis needs at least two frames")
        if st == K.WORLD_NONFINITE:
            raise ValueError("WORLD synthesis: f0, logspc or codeap holds NaN or inf")
        return wav[0, :int(wav_len[0])].double().cpu().numpy()
