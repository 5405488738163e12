"""Mel-cepstrum -> log-spectrum on the inference path (SURVEY.md section 8f #4).

The reference's shipped TTS config trains AlignTextToAudio on 25 mel-cepstral coefficients (config/tts_en_base.yaml:29
`vocoder: world_mcep`) and converts them back with a fixed matrix after `predict`
(voice100/export_onnx.py:81-97 `AlignTextToAudioPredict`, voice100/vocoder.py:115-123 `create_mc2sp_matrix`).
Un-normalisation and that matrix are both linear, so here they are folded into the projection layer: the head GEMM
emits the 257 log-spectrum bins directly and the conversion costs nothing at run time.
WORLD waveform synthesis itself (pyworld, a CPU C library) stays out of scope.
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
