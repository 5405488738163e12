"""TTS: TextToAlignTextModel and AlignTextToAudioModel (VoiceDecoder) on the libv100 kernels.

Interface mirrors voice100/models/tts.py:13-29,67-110,152-201 and WORLDNorm.unnormalize
(voice100/models/_layers_v1.py:96-138).  Inference only.
"""
from __future__ import annotations

from typing import Tuple

import torch
from torch import nn

from . import kernels as K
from ._lib import V100Error
from .blocks import (InvertedResidualParams, PreparedCache, StorageDtypeMixin, require_eval_cuda,
                     run_inverted_residual)
from .synth import ALIGN_KERNELS, VOICE_DECODER_POST_KERNELS, VOICE_DECODER_PRE_KERNELS

__all__ = ["TextToAlignTextModel", "AlignTextToAudioModel", "VoiceDecoder", "WORLDNorm", "align_batch", "TtsPipeline"]


def _head(conv: nn.Conv1d, dtype):
    return (conv.weight.detach()[:, :, 0].to(dtype).contiguous(), conv.bias.detach().float().contiguous())


class TextToAlignTextModel(StorageDtypeMixin, nn.Module):
    def __init__(self, vocab_size: int, hidden_size: int, learning_rate: float = 1e-3) -> None:
        super().__init__()
        self.hparams = dict(vocab_size=vocab_size, hidden_size=hidden_size, learning_rate=learning_rate)
        self.embedding = nn.Embedding(vocab_size, hidden_size)
        self.layers = nn.Sequential(
            *[InvertedResidualParams(hidden_size, hidden_size, k) for k in ALIGN_KERNELS],
            nn.Conv1d(hidden_size, 2, 1, bias=True))
        self._prepared = PreparedCache(self, lambda: dict(
            table=self.embedding.weight.detach().to(self.storage_dtype).contiguous(),
            blocks=[self.layers[i].prepare(self.storage_dtype) for i in range(4)],
            head=_head(self.layers[4], self.storage_dtype)))
        self.eval()

    def _head_ncw(self, x: torch.Tensor) -> K.Ncw:
        """text int64 [B, L] -> the head output as fp32 Ncw [B, 2, pitch] (rows: log(gap + 1), log(dur + 1))."""
        require_eval_cuda(self, x)
        w = self._prepared.get()
        h = K.embedding_ncw(x.contiguous(), w["table"])
        for blk in w["blocks"]:
            h = run_inverted_residual(h, blk)
        return K.conv1x1_f32(h, *w["head"])

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """text int64 [B, L] -> fp32 [B, L, 2] = log(align + 1)."""
        return K.ncw_f32_to_ntc(self._head_ncw(x))

    def align(self, text: torch.Tensor, align: torch.Tensor, head: int = 5, tail: int = 5) -> torch.Tensor:
        """Host-side expansion of one utterance's tokens to 20 ms frames (tts.py:89-110): token i fills
        frames [round(t + gap_i), round(t + gap_i + dur_i)), at least one; python round() semantics."""
        assert text.dim() == 1 and align.dim() == 2
        return torch.tensor(_align_one(text.detach().cpu().tolist(), align.detach().cpu().tolist(),
                                       head + int(torch.sum(align)) + tail, head), dtype=text.dtype)


def _align_one(toks, gaps, total: int, head: int):
    """The reference loop verbatim in its index behaviour (tts.py:100-110): `aligntext[j] = text[i]` on a tensor of
    `total` frames, so a NEGATIVE frame index wraps around from the end (a negative gap early in the text) and an
    index outside [-total, total) raises IndexError."""
    if total < 0:
        raise RuntimeError(f"Trying to create tensor with negative dimension {total}")   # torch.zeros(total) in the reference
    out = [0] * total
    t = head
    for (gap, dur), tok in zip(gaps, toks):
        t += gap
        s = round(t)
        t += dur
        e = round(t)
        if s == e:
            e = max(0, e + 1)
        for j in range(s, e):
            if j < -total or j >= total:
                raise IndexError(f"index {j} is out of bounds for dimension 0 with size {total}")
            out[j] = tok
    return out


def align_batch(text, align, text_len=None, head: int = 5, tail: int = 5, pad_value: int = 0):
    """Vectorised host form of `TextToAlignTextModel.align` over a padded batch: text int64 [B, L],
    align float [B, L, 2] (gap, duration per token, in 20 ms frames), optional text_len [B].
    -> (aligntext int64 [B, T_max] padded with `pad_value`, aligntext_len int32 [B]).
    Same arithmetic as the reference loop (tts.py:89-110): a float64 running sum of the float32 entries,
    round-half-to-even, every token at least one frame, total length head + int(sum(align)) + tail."""
    import numpy as np
    text_np = text.detach().cpu().numpy()
    al = align.detach().cpu().numpy().astype(np.float64)
    B, L = text_np.shape
    lens = np.full((B,), L, np.int64) if text_len is None else np.asarray(text_len.detach().cpu()).astype(np.int64)
    outs = []
    for b in range(B):
        n = int(lens[b])
        a = al[b, :n]
        flat = a.reshape(-1)                                  # gap0, dur0, gap1, dur1, ...
        t = head + np.cumsum(flat)                            # sequential double additions, like the loop
        s = np.rint(t[0::2]).astype(np.int64)                 # python round() == rint (half to even)
        e = np.rint(t[1::2]).astype(np.int64)
        e = np.where(s == e, np.maximum(0, e + 1), e)
        total = head + int(torch.sum(align[b, :n])) + tail    # the reference sums in float32 (torch.sum)
        if n and a.min() >= 0 and e.max() > total:
            raise IndexError("alignment runs past the aligned text (same failure as the reference)")
        if total < 0:
            raise RuntimeError(f"Trying to create tensor with negative dimension {total}")
        if n and (s.min() < 0 or a.min() < 0):
            # negative frame indices wrap around in the reference, and negative gaps / durations make the start frames
            # non-monotone: take the reference's own loop for this utterance
            outs.append(np.asarray(_align_one(text_np[b, :n].tolist(), a.tolist(), total, head), np.int64))
            continue
        # frame f belongs to the LAST token i with s_i <= f < e_i (later tokens overwrite earlier ones in the
        # reference loop); s is non-decreasing, so that is one searchsorted per utterance
        out = np.zeros((total,), np.int64)
        if n:
            f = np.arange(total)
            i = np.searchsorted(s, f, side="right") - 1
            ok = (i >= 0) & (f < e[np.maximum(i, 0)])
            out[ok] = text_np[b, i[ok]]
        outs.append(out)
    T = max(len(o) for o in outs)
    res = np.full((B, T), pad_value, np.int64)
    for b, o in enumerate(outs):
        res[b, :len(o)] = o
    return torch.from_numpy(res), torch.tensor([len(o) for o in outs], dtype=torch.int32)


class VoiceDecoder(StorageDtypeMixin, nn.Module):
    def __init__(self, hidden_size: int, out_channels: int) -> None:
        super().__init__()
        half = hidden_size // 2
        self.layers = nn.Sequential(
            *[InvertedResidualParams(hidden_size, hidden_size, k) for k in VOICE_DECODER_PRE_KERNELS],
            nn.ConvTranspose1d(hidden_size, half, kernel_size=5, padding=2, stride=2),
            *[InvertedResidualParams(half, half, k) for k in VOICE_DECODER_POST_KERNELS],
            nn.Conv1d(half, out_channels, 1, bias=True))
        self._prepared = PreparedCache(self, self._prepare)

    def _prepare(self):
        up = self.layers[4]
        c_in, c_out, _ = up.weight.shape
        # Wp[co][tap*C_in + ci] = weight[ci][co][tap]  (ConvTranspose1d stores [C_in, C_out, k])
        dtype = self.storage_dtype
        wp = up.weight.detach().permute(1, 2, 0).reshape(c_out, 5 * c_in).to(dtype).contiguous()
        return dict(pre=[self.layers[i].prepare(dtype) for i in range(4)], wp=wp,
                    up_bias=up.bias.detach().float().contiguous(),
                    post=[self.layers[i].prepare(dtype) for i in range(5, 8)], head=_head(self.layers[8], dtype))

    def run(self, x: K.Ncw) -> K.Ncw:
        """bf16 Ncw [B, H, T] -> fp32 Ncw [B, out_channels, 2T-1]."""
        w = self._prepared.get()
        for blk in w["pre"]:
            x = run_inverted_residual(x, blk)
        x = K.convtranspose_k5s2(x, w["wp"], w["up_bias"])
        for blk in w["post"]:
            x = run_inverted_residual(x, blk)
        return K.conv1x1_f32(x, *w["head"])

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        require_eval_cuda(self, x)
        return self.run(K.ncw_from_f32(x.float().contiguous(), self.storage_dtype)).valid().contiguous()


class WORLDNorm(nn.Module):
    """Per-feature mean/std of the WORLD parameters (_layers_v1.py:96-117); only `unnormalize` is on the
    inference path and it is fused into v100_world_finalize."""

    def __init__(self, logspc_size: int, codeap_size: int):
        super().__init__()
        mk = lambda v, n: nn.Parameter(torch.full([n], v), requires_grad=False)
        self.f0_std, self.f0_mean = mk(1.0, 1), mk(0.0, 1)
        self.logspc_std, self.logspc_mean = mk(1.0, logspc_size), mk(0.0, logspc_size)
        self.codeap_std, self.codeap_mean = mk(1.0, codeap_size), mk(0.0, codeap_size)

    def packed(self):
        mean = torch.cat([self.f0_mean, self.logspc_mean, self.codeap_mean]).detach().float().contiguous()
        std = torch.cat([self.f0_std, self.logspc_std, self.codeap_std]).detach().float().contiguous()
        return mean, std


class AlignTextToAudioModel(StorageDtypeMixin, nn.Module):
    def __init__(self, vocab_size: int, hidden_size: int, learning_rate: float = 1e-3, use_mcep: bool = False) -> None:
        super().__init__()
        self.hparams = dict(vocab_size=vocab_size, hidden_size=hidden_size, learning_rate=learning_rate,
                            use_mcep=use_mcep)
        self.hidden_size, self.vocab_size = hidden_size, vocab_size
        self.sample_rate, self.n_fft = 16000, 512
        # tts.py:164: 25 mel-cepstrum coefficients with use_mcep, else the n_fft // 2 + 1 log-spectrum bins
        self.hasf0_size, self.f0_size, self.logspc_size, self.codeap_size = 1, 1, (25 if use_mcep else 257), 1
        self.audio_size = self.hasf0_size + self.f0_size + self.logspc_size + self.codeap_size
        self.embedding = nn.Embedding(vocab_size, hidden_size)
        self.decoder = VoiceDecoder(hidden_size, self.audio_size)
        self.norm = WORLDNorm(self.logspc_size, self.codeap_size)
        self._prepared = PreparedCache(self, lambda: dict(
            table=self.embedding.weight.detach().to(self.storage_dtype).contiguous(), norm=self.norm.packed()))
        self.eval()

    def _decode(self, aligntext: torch.Tensor) -> K.Ncw:
        require_eval_cuda(self, aligntext)
        w = self._prepared.get()
        return self.decoder.run(K.embedding_ncw(aligntext.contiguous(), w["table"]))

    def forward(self, aligntext: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
        """aligntext int64 [B, T] -> (hasf0_logits [B,T'], f0_hat [B,T'], logspc_hat [B,T',logspc_size],
        codeap_hat [B,T',1]) normalised, T' = 2T-1."""
        return K.world_finalize(self._decode(aligntext), None, None, False, self.logspc_size, self.codeap_size, 1)

    def predict(self, aligntext: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """-> (f0 [B,T'], logspc [B,T',logspc_size], codeap [B,T',1]) un-normalised, f0 = 0 where unvoiced."""
        y = self._decode(aligntext)
        mean, std = self._prepared.get()["norm"]
        _, f0, logspc, codeap = K.world_finalize(y, mean, std, True, self.logspc_size, self.codeap_size, 1)
        return f0, logspc, codeap


class TtsPipeline:
    """text -> WORLD parameters for TextToAlignTextModel + AlignTextToAudioModel, every stage a libv100 kernel and
    the alignment on the device (v100_tts_align): align model -> exp(pred) - 1 and the frame expansion of
    TextToAlignTextModel.align in one kernel -> audio model -> WORLD parameters.  Same results, bit for bit, as the
    stepwise composition `align_model(text)` -> `torch.exp(pred) - 1` -> `align_batch` -> `audio_model.predict`.

    `pipe(text, text_len=None, max_frames=None)` -> (f0 [B,T'], logspc [B,T',S], codeap [B,T',A], frame_len int32 [B],
    status int32 [B]); frame_len = 2 * aligned length - 1 valid WORLD frames (0 for a failed utterance), status the
    V100_ALIGN_* code (kernels.ALIGN_*).  Without `max_frames` the aligned text is sized to the batch's longest
    utterance (one small host round trip) and an utterance the host loop fails on raises its exception; with
    `max_frames` nothing waits on the host and nothing raises: utterances longer than max_frames frames are cut
    (ALIGN_CAPACITY) and failed ones come back with frame_len 0.  `.graphed()` captures the whole path into one CUDA
    graph.  The v1 models see the whole [B, L] text whatever `text_len` says (the reference's own behaviour):
    text_len only limits which tokens are expanded into frames."""
    rule = 1

    def __init__(self, align_model, audio_model, head: int = 5, tail: int = 5):
        self.align_model, self.audio_model, self.head, self.tail = align_model, audio_model, head, tail

    def _durations(self, text: torch.Tensor, text_len):
        """-> fp32 [B, L, 2] log(1 + (gap, duration)): a strided view of the head output, read in place."""
        y = self.align_model._head_ncw(text)
        return y.data.transpose(1, 2)[:, :text.shape[1]]

    def _audio(self, aligntext: torch.Tensor, filled_len: torch.Tensor):
        return self.audio_model.predict(aligntext)

    @torch.no_grad()
    def __call__(self, text: torch.Tensor, text_len: torch.Tensor = None, max_frames: int = None):
        dev = next(self.align_model.parameters()).device
        text = text.to(dev)
        if text_len is not None:
            text_len = text_len.to(device=dev, dtype=torch.int32)
        pred = self._durations(text, text_len)
        if max_frames is None:
            at, lens = K._align_exact(text, pred, text_len, self.rule, self.head, self.tail, True)
        else:
            at, lens = K.tts_align(text, pred, text_len, self.rule, self.head, self.tail, int(max_frames), True)
        f0, logspc, codeap = self._audio(at, lens[2])
        return f0, logspc, codeap, lens[3], lens[1]

    @torch.no_grad()
    def graphed(self, batch: int, text_len_max: int, max_frames: int, device="cuda"):
        """Capture text -> WORLD parameters for [batch, text_len_max] token ids and `max_frames` aligned frames into one
        CUDA graph.  Returns `run(text, text_len=None) -> (f0, logspc, codeap, frame_len, status)`: `text` must be
        [batch, text_len_max]; the outputs are static buffers overwritten by the next replay, and equal bit for bit
        what `pipe(text, text_len, max_frames)` returns eagerly."""
        dev = torch.device(device)
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        with torch.cuda.device(dev):
            text_s = torch.zeros((batch, text_len_max), dtype=torch.int64, device=dev)
            len_s = torch.full((batch,), text_len_max, dtype=torch.int32, device=dev)
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):          # warm-up outside capture: prepared weights, function attributes
                for _ in range(2):
                    self(text_s, len_s, max_frames)
            torch.cuda.current_stream(dev).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                outs = self(text_s, len_s, max_frames)

        def run(text: torch.Tensor, text_len: torch.Tensor = None):
            if tuple(text.shape) != (batch, text_len_max):
                raise V100Error(f"graphed TTS pipeline: text must be [{batch}, {text_len_max}], got {tuple(text.shape)}")
            text_s.copy_(text, non_blocking=True)
            if text_len is None:
                len_s.fill_(text_len_max)
            else:
                len_s.copy_(text_len, non_blocking=True)
            graph.replay()
            return outs
        run.graph, run.text, run.text_len, run.outputs = graph, text_s, len_s, outs
        return run
