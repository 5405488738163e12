"""The v2 models of the reference -- what its shipped configs and released checkpoints are -- on libv100:

  AudioToAlignText   voice100/models/_asr_v2.py:18-49    conv blocks -> 2-layer biLSTM -> Linear (CTC logits)
  TextToAlignText    voice100/models/_align_v2.py:17-82  Embedding -> 2-layer biLSTM -> Linear (log durations)
  AlignTextToAudio   voice100/models/_tts_v2.py:13-91    Embedding -> biLSTM -> conv / transposed-conv blocks -> WORLD
  ConvLayerBlock / ConvTransposeLayerBlock / get_conv_layers   voice100/models/_layers_v2.py:29-103

Same constructor arguments, call signatures and `state_dict` keys as the reference (stock nn.Conv1d /
nn.LayerNorm / nn.LSTM / nn.Linear objects hold the parameters; their own forward is never used).  Inference only.

Data flow: conv blocks run on the NCW layout of the v1 path; around the recurrent layers activations are
time-major (kernels.Tm), so that each layer's input projection is one GEMM over all steps and the recurrence
is one persistent kernel per layer (v100_lstm_layer).
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import torch
from torch import nn

from . import kernels as K
from ._lib import V100Error
from .asr import AsrPipeline
from .blocks import PreparedCache, StorageDtypeMixin, require_eval_cuda
from .tts import TtsPipeline, WORLDNorm

__all__ = ["ConvLayerBlock", "ConvTransposeLayerBlock", "get_conv_layers", "AudioToAlignText", "TextToAlignText",
           "AlignTextToAudio", "AsrV2Pipeline", "align_batch_v2", "TtsV2Pipeline"]


class ConvLayerBlock(nn.Module):
    """Conv1d -> LayerNorm(channels) -> GELU (_layers_v2.py:29-57)."""
    transpose = False

    def __init__(self, in_channels: int, out_channels: int, kernel_size: int, stride: int, padding: int, bias: bool):
        super().__init__()
        self.layer_norm = nn.LayerNorm(normalized_shape=out_channels)
        self.conv = nn.Conv1d(in_channels, out_channels, kernel_size, stride=stride, padding=padding, bias=bias)

    def forward(self, *a, **k):  # pragma: no cover
        raise V100Error("ConvLayerBlock holds parameters only; it runs through get_conv_layers(...).run")

    def prepare(self, dtype):
        w = self.conv.weight.detach()
        c_out, c_in, k = w.shape
        if (k * c_in) % 8 != 0:
            raise V100Error(f"ConvLayerBlock: kernel_size*in_channels = {k * c_in} must be a multiple of 8")
        bias = self.conv.bias.detach().float() if self.conv.bias is not None else torch.zeros(c_out, device=w.device)
        return dict(transpose=False, k=k, stride=self.conv.stride[0], pad=self.conv.padding[0],
                    wp=w.permute(0, 2, 1).reshape(c_out, k * c_in).to(dtype).contiguous(),   # [co][tap*C_in + ci]
                    bias=bias.contiguous(), gamma=self.layer_norm.weight.detach().float().contiguous(),
                    beta=self.layer_norm.bias.detach().float().contiguous(), eps=self.layer_norm.eps)


class ConvTransposeLayerBlock(nn.Module):
    """ConvTranspose1d -> LayerNorm(channels) -> GELU (_layers_v2.py:60-88)."""
    transpose = True

    def __init__(self, in_channels: int, out_channels: int, kernel_size: int, stride: int, padding: int, bias: bool):
        super().__init__()
        if (kernel_size, stride, padding) != (5, 2, 2):
            raise V100Error("ConvTransposeLayerBlock: only kernel_size=5, stride=2, padding=2 (the shipped configs) "
                            "is on the accelerated path")
        self.layer_norm = nn.LayerNorm(normalized_shape=out_channels)
        self.conv = nn.ConvTranspose1d(in_channels, out_channels, kernel_size, stride=stride, padding=padding,
                                       bias=bias)

    def forward(self, *a, **k):  # pragma: no cover
        raise V100Error("ConvTransposeLayerBlock holds parameters only; it runs through get_conv_layers(...).run")

    def prepare(self, dtype):
        w = self.conv.weight.detach()                    # [C_in, C_out, 5]
        c_in, c_out, _ = w.shape
        bias = self.conv.bias.detach().float() if self.conv.bias is not None else torch.zeros(c_out, device=w.device)
        return dict(transpose=True, wp=w.permute(1, 2, 0).reshape(c_out, 5 * c_in).to(dtype).contiguous(),
                    bias=bias.contiguous(), gamma=self.layer_norm.weight.detach().float().contiguous(),
                    beta=self.layer_norm.bias.detach().float().contiguous(), eps=self.layer_norm.eps)


class ConvLayers(StorageDtypeMixin, nn.Sequential):
    """nn.Sequential of the blocks (so the keys are `{i}.conv.*`, `{i}.layer_norm.*`) plus the libv100 runner."""

    def __init__(self, *blocks):
        super().__init__(*blocks)
        self._prepared = PreparedCache(self, lambda: [b.prepare(self.storage_dtype) for b in self])

    def run(self, x: K.Ncw) -> K.Ncw:
        for w in self._prepared.get():
            if w["transpose"]:
                x = K.convtranspose_k5s2(x, w["wp"], w["bias"])
            else:
                x = K.conv1d(x, w["wp"], w["bias"], w["k"], w["stride"], w["pad"])
            x = K.layernorm_gelu(x, w["gamma"], w["beta"], w["eps"])
        return x

    def run_to_tm(self, x: K.Ncw) -> K.Tm:
        """Same blocks, result in the time-major layout the recurrent layers want.  The trailing run of stride-1
        "same"-padded convolutions is evaluated ON the time-major tensor (v100_conv1d_tm: taps are aligned column
        offsets, no tap stack); the layout change happens in front of it."""
        ws = self._prepared.get()
        n_tm = 0
        for w in reversed(ws):
            if w["transpose"] or w["stride"] != 1 or 2 * w["pad"] + 1 != w["k"] or w["k"] > 5 or \
                    (w["wp"].shape[1] // w["k"]) % 64 != 0:
                break
            n_tm += 1
        for w in ws[:len(ws) - n_tm]:
            if w["transpose"]:
                x = K.convtranspose_k5s2(x, w["wp"], w["bias"])
            else:
                x = K.conv1d(x, w["wp"], w["bias"], w["k"], w["stride"], w["pad"])
            x = K.layernorm_gelu(x, w["gamma"], w["beta"], w["eps"])
        tm = K.ncw_to_tm(x)
        for w in ws[len(ws) - n_tm:]:
            tm = K.layernorm_gelu_tm(K.conv1d_tm(tm, w["wp"], w["bias"], w["k"]), w["gamma"], w["beta"], w["eps"])
        return tm

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """fp32 [B, C, T] -> fp32 [B, C', T'] (module-level parity with the reference's nn.Sequential)."""
        require_eval_cuda(self, x)
        return K.ncw_to_f32(self.run(K.ncw_from_f32(x.float().contiguous(), self.storage_dtype)))


def get_conv_layers(in_channels: int, settings: Sequence[Sequence]) -> ConvLayers:
    """settings rows: (out_channels, transpose, kernel_size, stride, padding, bias) -- _layers_v2.py:91-103."""
    blocks, c = [], in_channels
    for out_channels, transpose, kernel_size, stride, padding, bias in settings:
        cls = ConvTransposeLayerBlock if transpose else ConvLayerBlock
        blocks.append(cls(c, out_channels, kernel_size=kernel_size, stride=stride, padding=padding, bias=bias))
        c = out_channels
    return ConvLayers(*blocks)


def _prepare_lstm(lstm: nn.LSTM, dtype) -> List[dict]:
    """Per layer: w_ih [8H, I] (forward rows first), bias fp32 [8H] = b_ih + b_hh, w_hh [2, 4H, H]."""
    if not lstm.bidirectional or lstm.proj_size != 0 or not lstm.bias:
        raise V100Error("only bidirectional nn.LSTM with bias and without projection is on the accelerated path")
    out = []
    for n in range(lstm.num_layers):
        def g(name):
            return getattr(lstm, f"{name}_l{n}").detach(), getattr(lstm, f"{name}_l{n}_reverse").detach()
        w_ih = torch.cat(g("weight_ih"), 0).to(dtype).contiguous()
        w_hh = torch.stack(g("weight_hh"), 0).to(dtype).contiguous()
        bias = (torch.cat(g("bias_ih"), 0).float() + torch.cat(g("bias_hh"), 0).float()).contiguous()
        out.append(dict(w_ih=w_ih, w_hh=w_hh, bias=bias))
    return out


def _run_lstm(x: K.Tm, layers: List[dict], lengths: torch.Tensor) -> K.Tm:
    lengths = lengths.to(device=x.data.device, dtype=torch.int32).contiguous()
    ws = K.lstm_workspace(x.B, layers[0]["w_hh"].shape[2], x.data.device)
    for w in layers:
        x = K.lstm_layer(x, w["w_ih"], w["bias"], w["w_hh"], lengths, ws)
    return x


def _head(lin: nn.Linear, dtype):
    return lin.weight.detach().to(dtype).contiguous(), lin.bias.detach().float().contiguous()


def _tm_head_to_tbc(y: K.Ncw, tm: K.Tm) -> torch.Tensor:
    """fp32 head output over a time-major tensor ([1, C, T*Bp]) -> [T, B, C]."""
    out = K.ncw_f32_to_ntc(y)                            # [1, T*Bp, C]
    return out.view(tm.T, tm.Bp, y.C)[:, :tm.B]


class AudioToAlignText(StorageDtypeMixin, nn.Module):
    """CTC acoustic model of the shipped asr_*.yaml configs (_asr_v2.py:18-49)."""

    def __init__(self, audio_size: int, encoder_settings: List[List], decoder_num_layers: int,
                 decoder_hidden_size: int, vocab_size: int, learning_rate: float = 0.001) -> None:
        super().__init__()
        self.hparams = dict(audio_size=audio_size, encoder_settings=encoder_settings,
                            decoder_num_layers=decoder_num_layers, decoder_hidden_size=decoder_hidden_size,
                            vocab_size=vocab_size, learning_rate=learning_rate)
        self.encoder = get_conv_layers(audio_size, encoder_settings)
        self.lstm = nn.LSTM(input_size=decoder_hidden_size, hidden_size=decoder_hidden_size,
                            num_layers=decoder_num_layers, dropout=0.2, bidirectional=True)
        self.dense = nn.Linear(decoder_hidden_size * 2, vocab_size)
        self._prepared = PreparedCache(self, lambda: dict(lstm=_prepare_lstm(self.lstm, self.storage_dtype),
                                                          head=_head(self.dense, self.storage_dtype)))
        self.eval()

    @staticmethod
    def output_length(audio_len: torch.Tensor) -> torch.Tensor:
        return torch.div(audio_len + 1, 2, rounding_mode="trunc")          # _asr_v2.py:43

    def _run(self, x: K.Ncw, x_len: torch.Tensor):
        """16-bit Ncw features -> (fp32 head output over the time-major tensor, that tensor's geometry)."""
        w = self._prepared.get()
        tm = _run_lstm(self.encoder.run_to_tm(x), w["lstm"], x_len)
        return K.conv1x1_f32(tm.as_ncw(), *w["head"]), tm

    def forward(self, audio: torch.Tensor, audio_len: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """audio fp32 [B, T, audio_size], audio_len [B] -> (logits fp32 [T', B, V] time-major, lengths [B]) with
        T' = max length, as pad_packed_sequence(batch_first=False) returns them (_asr_v2.py:47-49)."""
        require_eval_cuda(self, audio)
        x_len = self.output_length(audio_len.to(audio.device))
        y, tm = self._run(K.ntc_f32_to_ncw(audio.float().contiguous(), self.storage_dtype), x_len)
        t_max = min(int(x_len.max()), tm.T)
        return _tm_head_to_tbc(y, tm)[:t_max].contiguous(), x_len.cpu()

    def greedy(self, audio, audio_len: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """argmax tokens int64 [T', B] (T' = padded length, no host sync) and lengths [B] on the device; what
        ctc_best_path(text=None) returns (_asr_v2.py:95-96).  `audio` fp32 [B, T, 64] or a 16-bit Ncw from logmel."""
        if not isinstance(audio, K.Ncw):
            require_eval_cuda(self, audio)
            audio = K.ntc_f32_to_ncw(audio.float().contiguous(), self.storage_dtype)
        x_len = self.output_length(audio_len.to(audio.data.device))
        y, tm = self._run(audio, x_len)
        _, tokens = K.ctc_finalize(y, want_logits=False)           # [1, T*Bp]
        return tokens.view(tm.T, tm.Bp)[:, :tm.B], x_len


def _ctc_best_path_method(self, audio: torch.Tensor = None, audio_len: torch.Tensor = None,
                          text: torch.Tensor = None, text_len: torch.Tensor = None, logits: torch.Tensor = None):
    """AudioToAlignText.ctc_best_path (_asr_v2.py:84-119), the core of `voice100-align-text`, with the per-utterance
    numpy DP replaced by the batched Viterbi kernel.  text is None -> argmax tokens [T', B] (what the reference
    returns); otherwise -> (score fp32 [B], hist int32 [B, T'] = state index per frame, path int64 [B, T'] =
    expanded label per frame, logits_len [B]).  (The reference's `score` output is overwritten by a leftover
    variable, _asr_v2.py:116; here it is the best-path log-probability.)"""
    from .align import ctc_best_path_batch
    normalize = logits is None      # fresh logits: log_softmax (_asr_v2.py:95) is folded into the Viterbi kernel
    if logits is None:
        logits, logits_len = self.forward(audio, audio_len)
    else:
        logits_len = audio_len
    if text is None:
        return logits.argmax(dim=-1)                                          # argmax is invariant under log_softmax
    dev = logits.device
    logits_len = logits_len.to(dev)
    text_len = torch.minimum(logits_len, text_len.to(dev))                    # "for very short audio", :99
    return ctc_best_path_batch(logits.transpose(0, 1).contiguous(), logits_len.to(torch.int32), text.to(dev),
                               text_len.to(torch.int32), normalize=normalize)


AudioToAlignText.ctc_best_path = torch.no_grad()(_ctc_best_path_method)


class AsrV2Pipeline(AsrPipeline):
    """waveform -> tokens for AudioToAlignText: log-mel, conv blocks, LSTM stack, head and argmax on libv100.
    Same interface as AsrPipeline -- `pipe(waveform, lengths) -> (tokens int64 [B, T'], lengths [B])`, `.graphed()`,
    `.submit_host()/.transcribe_host()` (pinned-host streaming on two alternating buffer sets), `.transcribe_ids()`;
    `model.greedy` keeps the reference's time-major [T', B] form."""

    def __init__(self, transform, model: AudioToAlignText):
        self.transform, self.model = transform, model

    @torch.no_grad()
    def __call__(self, waveform: torch.Tensor, lengths: torch.Tensor):
        feats, audio_len = self.transform.logmel_batch(waveform, lengths, ncw_dtype=self.model.storage_dtype)
        tokens, x_len = self.model.greedy(feats, audio_len)
        return tokens.t().contiguous(), x_len


class TextToAlignText(StorageDtypeMixin, nn.Module):
    """Duration model of align_*.yaml (_align_v2.py:17-82)."""

    def __init__(self, vocab_size, num_layers, hidden_size, num_outputs, learning_rate=1e-3) -> None:
        super().__init__()
        assert num_outputs == 2
        self.hparams = dict(vocab_size=vocab_size, num_layers=num_layers, hidden_size=hidden_size,
                            num_outputs=num_outputs, learning_rate=learning_rate)
        self.embedding = nn.Embedding(vocab_size, hidden_size)
        self.lstm = nn.LSTM(input_size=hidden_size, hidden_size=hidden_size, num_layers=num_layers, dropout=0.2,
                            bidirectional=True, batch_first=True)
        self.dense = nn.Linear(hidden_size * 2, num_outputs)
        self._prepared = PreparedCache(self, lambda: dict(
            table=self.embedding.weight.detach().to(self.storage_dtype).contiguous(),
            lstm=_prepare_lstm(self.lstm, self.storage_dtype), head=_head(self.dense, self.storage_dtype)))
        self.eval()

    def _head_tm(self, text: torch.Tensor, text_len: torch.Tensor):
        """-> (fp32 head output over the time-major tensor, [1, 2, T*Bp] with column t*Bp + b, that tensor's
        geometry); no host synchronisation."""
        require_eval_cuda(self, text)
        w = self._prepared.get()
        tm = K.ncw_to_tm(K.embedding_ncw(text.contiguous(), w["table"]))
        tm = _run_lstm(tm, w["lstm"], text_len)
        return K.conv1x1_f32(tm.as_ncw(), *w["head"]), tm

    def forward(self, text: torch.Tensor, text_len: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """text int64 [B, L], text_len [B] -> (fp32 [B, max_len, 2], lengths) (_align_v2.py:29-43)."""
        y, tm = self._head_tm(text, text_len)
        y = _tm_head_to_tbc(y, tm)
        t_max = min(int(text_len.max()), tm.T)
        return y[:t_max].transpose(0, 1).contiguous(), text_len.cpu()

    def predict(self, text: torch.Tensor, text_len: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        align, align_len = self.forward(text, text_len)
        return torch.exp(align) - 1, align_len

    @staticmethod
    def align(text: torch.Tensor, align: torch.Tensor, head=5, tail=5) -> torch.Tensor:
        """Host-side expansion of one utterance (_align_v2.py:54-82): truncating frame positions, the first token's
        gap ignored, at least one blank frame before and one frame for every token."""
        assert text.dim() == 1 and align.dim() == 2
        a = align.detach().cpu()
        n = head + int(torch.sum(a) - a[0, 0]) + tail
        out = torch.zeros(n, dtype=text.dtype)
        t, u = head, 0
        gap, dur = a[:, 0].tolist(), a[:, 1].tolist()
        toks = text.detach().cpu().tolist()
        for i in range(a.shape[0]):
            if i > 0:
                t += gap[i]
            s = max(int(t), u)
            u = s + 1
            t += dur[i]
            e = max(int(t), u)
            u = e
            out[s:e] = toks[i]
        return out


def align_batch_v2(text, align, text_len=None, head: int = 5, tail: int = 5, pad_value: int = 0):
    """`TextToAlignText.align` (_align_v2.py:54-82) over a padded batch on the host: text int64 [B, L], align float
    [B, L, 2], optional text_len [B] -> (aligntext int64 [B, T_max], aligntext_len int32 [B]).  Same arithmetic as the
    reference loop: float64 running sum of the float32 entries with the first gap skipped, int() truncation,
    s_i = max(int(t), e_{i-1}), e_i = max(int(t + dur_i), s_i + 1)."""
    import numpy as np
    text_np = text.detach().cpu().numpy()
    al32 = align.detach().cpu()
    al = al32.numpy().astype(np.float64)
    B, L = text_np.shape
    lens = np.full((B,), L, np.int64) if text_len is None else np.asarray(text_len.detach().cpu()).astype(np.int64)
    flat = al.reshape(B, 2 * L).copy()
    flat[:, 0] = 0.0                                          # the first token's gap is not applied
    t = head + np.cumsum(flat, axis=1)
    a, b = t[:, 0::2].astype(np.int64), t[:, 1::2].astype(np.int64)
    s, e = np.empty_like(a), np.empty_like(b)
    prev = np.zeros((B,), np.int64)
    for i in range(L):                                        # running max: sequential in i, vector over the batch
        s[:, i] = np.maximum(a[:, i], prev)
        e[:, i] = np.maximum(b[:, i], s[:, i] + 1)
        prev = e[:, i]
    outs = []
    for u in range(B):
        n = int(lens[u])
        total = head + int(torch.sum(al32[u, :n]) - al32[u, 0, 0]) + tail if n else head + tail
        if n and e[u, n - 1] > total:
            raise IndexError("alignment runs past the aligned text (same failure as the reference)")
        out = np.zeros((total,), np.int64)
        if n:
            seg = e[u, :n] - s[u, :n]
            pos = np.repeat(s[u, :n] - (np.cumsum(seg) - seg), seg) + np.arange(int(seg.sum()))
            out[pos] = np.repeat(text_np[u, :n], seg)
        outs.append(out)
    T = max(len(o) for o in outs)
    res = np.full((B, T), pad_value, np.int64)
    for u, o in enumerate(outs):
        res[u, :len(o)] = o
    return torch.from_numpy(res), torch.tensor([len(o) for o in outs], dtype=torch.int32)


class AlignTextToAudio(StorageDtypeMixin, nn.Module):
    """WORLD-parameter synthesiser of tts_*.yaml (_tts_v2.py:13-91)."""

    def __init__(self, vocab_size: int, logspc_size: int, codeap_size: int, encoder_num_layers: int,
                 encoder_hidden_size: int, decoder_settings: List[List], logspc_weight: float = 5.0,
                 learning_rate: float = 1e-3, f0_size: int = 1, audio_stat=None) -> None:
        super().__init__()
        self.hparams = dict(vocab_size=vocab_size, logspc_size=logspc_size, codeap_size=codeap_size,
                            encoder_num_layers=encoder_num_layers, encoder_hidden_size=encoder_hidden_size,
                            decoder_settings=decoder_settings, logspc_weight=logspc_weight,
                            learning_rate=learning_rate, f0_size=f0_size, audio_stat=audio_stat)
        assert f0_size == 1
        self.encoder_hidden_size, self.vocab_size = encoder_hidden_size, vocab_size
        self.f0_size, self.logspc_size, self.codeap_size = f0_size, logspc_size, codeap_size
        self.audio_size = 2 * f0_size + logspc_size + 2 * codeap_size
        self.embedding = nn.Embedding(vocab_size, encoder_hidden_size)
        self.lstm = nn.LSTM(input_size=encoder_hidden_size, hidden_size=encoder_hidden_size,
                            num_layers=encoder_num_layers, dropout=0.2, bidirectional=True)
        self.decoder = get_conv_layers(2 * encoder_hidden_size, decoder_settings)
        self.projection = nn.Linear(decoder_settings[-1][0], self.audio_size)
        self.norm = WORLDNorm(logspc_size, codeap_size)
        if audio_stat is not None:
            self.norm.load_state_dict(torch.load(audio_stat))
        self._prepared = PreparedCache(self, lambda: dict(
            table=self.embedding.weight.detach().to(self.storage_dtype).contiguous(),
            lstm=_prepare_lstm(self.lstm, self.storage_dtype), head=_head(self.projection, self.storage_dtype),
            norm=self.norm.packed()))
        self.eval()

    def _decode(self, aligntext: torch.Tensor, aligntext_len: torch.Tensor, t_max: int = None) -> K.Ncw:
        """`t_max` (default: the longest length, read back from the device) = the steps the LSTM runs over."""
        require_eval_cuda(self, aligntext)
        w = self._prepared.get()
        if t_max is None:
            t_max = int(aligntext_len.max())             # pad_packed_sequence trims to the longest utterance
        tm = K.ncw_to_tm(K.embedding_ncw(aligntext[:, :t_max].contiguous(), w["table"]))
        tm = _run_lstm(tm, w["lstm"], aligntext_len)
        x = self.decoder.run(K.tm_to_ncw(tm))
        return K.conv1x1_f32(x, *w["head"])              # fp32 Ncw [B, audio_size, T']

    def forward(self, aligntext: torch.Tensor, aligntext_len: torch.Tensor):
        """aligntext int64 [B, T], lengths [B] -> (hasf0_logits [B,T'], f0_hat [B,T'], logspc_hat [B,T',S],
        hascodeap_logits [B,T',A], codeap_hat [B,T',A]), T' = 2*max(len) - 1 for the shipped decoder."""
        return K.world_finalize(self._decode(aligntext, aligntext_len), None, None, False, self.logspc_size,
                                self.codeap_size, 2)

    def predict(self, aligntext: torch.Tensor, aligntext_len: torch.Tensor, t_max: int = None):
        """-> (f0 [B,T'], logspc [B,T',S], codeap [B,T',A]) un-normalised; f0 / codeap zeroed where their presence
        logits are negative (_tts_v2.py:80-91) -- split, WORLDNorm.unnormalize and both `where`s in one kernel.
        `t_max`: decode the first t_max frames without reading the lengths back (default max(aligntext_len))."""
        y = self._decode(aligntext, aligntext_len, t_max)
        mean, std = self._prepared.get()["norm"]
        _, f0, logspc, _, codeap = K.world_finalize(y, mean, std, True, self.logspc_size, self.codeap_size, 2)
        return f0, logspc, codeap


class TtsV2Pipeline(TtsPipeline):
    """text -> WORLD parameters for TextToAlignText + AlignTextToAudio (or AlignTextToAudioPredict, the form the shipped
    mel-cepstral tts_en_base.yaml needs): LSTM duration model -> exp(pred) - 1 and the frame expansion of
    TextToAlignText.align in one kernel (v100_tts_align, reading the head output over the time-major tensor in place)
    -> audio model -> WORLD parameters.  Same results, bit for bit, as `TextToAlignText.predict` -> `align_batch_v2` ->
    `AlignTextToAudio.predict` wherever align_batch_v2 does not raise; where it raises because a token runs past the
    total length, this follows `TextToAlignText.align` and drops those frames.  Same interface as TtsPipeline.

    With `max_frames` the audio model's LSTM runs max_frames steps whatever the utterances' lengths (a captured graph
    has fixed shapes).  A step is latency-bound and costs about 4 us, so keep the capacity close to the expected
    longest utterance."""
    rule = 2

    def _durations(self, text: torch.Tensor, text_len):
        if text_len is None:
            text_len = torch.full((text.shape[0],), text.shape[1], dtype=torch.int32, device=text.device)
        y, tm = self.align_model._head_tm(text, text_len)
        return torch.as_strided(y.data, (tm.B, tm.T, 2), (1, tm.Bp, y.pitch))

    def _audio(self, aligntext: torch.Tensor, filled_len: torch.Tensor):
        m = self.audio_model
        return (m.predict if isinstance(m, AlignTextToAudio) else m)(aligntext, filled_len, t_max=aligntext.shape[1])
