"""ASR: ConvVoiceEncoder + LinearCharDecoder + CTC greedy, on the libv100 kernels.

Interface mirrors voice100/models/asr.py:62-122 (constructor arguments, `forward`, `output_length`,
`.encoder` / `.decoder` sub-modules working on NCW tensors, `state_dict` keys).  Inference only.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import nn

from . import kernels as K
from ._lib import V100Error
from .data_modules import resampled_length
from .blocks import (InvertedResidualParams, PreparedCache, StorageDtypeMixin, require_eval_cuda,
                     run_inverted_residual)
from .synth import asr_encoder_blocks

__all__ = ["AudioToTextCTC", "ConvVoiceEncoder", "LinearCharDecoder"]


class ConvVoiceEncoder(StorageDtypeMixin, nn.Module):
    def __init__(self, in_channels: int, out_channels: int, hidden_size: int):
        super().__init__()
        self.layers = nn.Sequential(*[
            InvertedResidualParams(ci, co, k, s, r)
            for ci, co, k, s, r in asr_encoder_blocks(in_channels, out_channels, hidden_size)])
        self._prepared = PreparedCache(self, lambda: [blk.prepare(self.storage_dtype) for blk in self.layers])

    def run(self, x: K.Ncw) -> K.Ncw:
        for w in self._prepared.get():
            x = run_inverted_residual(x, w)
        return x

    def forward(self, embed: torch.Tensor) -> torch.Tensor:
        """fp32 NCW [B, in_channels, T] -> fp32 NCW [B, out_channels, (T+1)//2]."""
        require_eval_cuda(self, embed)
        return K.ncw_to_f32(self.run(K.ncw_from_f32(embed.float().contiguous(), self.storage_dtype)))

    def output_length(self, embed_len: torch.Tensor) -> torch.Tensor:
        return torch.div(embed_len + 1, 2, rounding_mode="trunc")


class LinearCharDecoder(StorageDtypeMixin, nn.Module):
    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        # index 0 is Dropout(0.2) in the reference (identity in eval); index 1 carries the weights
        self.layers = nn.Sequential(nn.Identity(), nn.Conv1d(in_channels, out_channels, 1, bias=True))
        self._prepared = PreparedCache(self, lambda: (
            self.layers[1].weight.detach()[:, :, 0].to(self.storage_dtype).contiguous(),
            self.layers[1].bias.detach().float().contiguous()))

    def run(self, x: K.Ncw) -> K.Ncw:
        W, b = self._prepared.get()
        return K.conv1x1_f32(x, W, b)

    def forward(self, enc_out: torch.Tensor) -> torch.Tensor:
        """fp32 NCW [B, embed, T] -> fp32 NCW logits [B, V, T]."""
        require_eval_cuda(self, enc_out)
        y = self.run(K.ncw_from_f32(enc_out.float().contiguous(), self.storage_dtype))
        return y.valid().contiguous()


class AudioToTextCTC(StorageDtypeMixin, nn.Module):
    def __init__(self, audio_size: int, embed_size: int, vocab_size: int, hidden_size: int,
                 learning_rate: float = 1e-3, weight_decay: float = 0.0):
        super().__init__()
        self.hparams = dict(audio_size=audio_size, embed_size=embed_size, vocab_size=vocab_size,
                            hidden_size=hidden_size, learning_rate=learning_rate, weight_decay=weight_decay)
        self.embed_size = embed_size
        self.encoder = ConvVoiceEncoder(audio_size, embed_size, hidden_size)
        self.decoder = LinearCharDecoder(embed_size, vocab_size)
        self.eval()

    def _run(self, x: K.Ncw, want_logits: bool, audio_len: torch.Tensor = None):
        return K.ctc_finalize(self.decoder.run(self.encoder.run(x)), want_logits, audio_len)

    def forward(self, audio: torch.Tensor) -> torch.Tensor:
        """audio fp32 [B, T, audio_size] -> logits fp32 [B, (T+1)//2, vocab_size]."""
        require_eval_cuda(self, audio)
        return self._run(K.ntc_f32_to_ncw(audio.float().contiguous(), self.storage_dtype), True)[0]

    def greedy(self, audio, audio_len: torch.Tensor = None):
        """CTC best-path tokens int64 [B, (T+1)//2] = forward(audio).argmax(-1) without materialising the
        logits.  `audio` is fp32 [B, T, 64] or the bf16 Ncw produced by logmel_batch(ncw_bf16=True).
        With `audio_len` (int32 [B] on the device) -> (tokens, output_length(audio_len)), both from one kernel."""
        if isinstance(audio, K.Ncw):
            require_eval_cuda(self, audio.data)
            x = audio
        else:
            require_eval_cuda(self, audio)
            x = K.ntc_f32_to_ncw(audio.float().contiguous(), self.storage_dtype)
        out = self._run(x, False, audio_len)
        return out[1] if audio_len is None else (out[1], out[2])

    def output_length(self, audio_len: torch.Tensor) -> torch.Tensor:
        return self.encoder.output_length(audio_len)


class AsrPipeline:
    """waveform -> tokens: log-mel + encoder + CTC head + greedy argmax, every stage a libv100 kernel.
    This is the path BASELINE.json's metric (ASR audio-seconds/second) is measured on."""

    def __init__(self, transform, model: AudioToTextCTC):
        self.transform, self.model = transform, model

    def _rate(self, sample_rate):
        """The input rate as a resampling key: None when it is the transform's own rate (no resampling)."""
        return None if sample_rate is None or sample_rate == self.transform.sample_rate else sample_rate

    @torch.no_grad()
    def __call__(self, waveform: torch.Tensor, lengths: torch.Tensor,
                 sample_rate: Optional[int] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """device waveform fp32 or int16 PCM [B, L], lengths [B] -> (tokens int64 [B, T'], valid lengths int32 [B]).
        Three kinds of kernel and nothing else: log-mel (also emits audio_len), the conv stack, the CTC tail (also
        emits output_length).  `sample_rate` is the waveform's rate (None = the transform's); any other rate is
        resampled on the device first (one more kernel: MelSpectrogramAudioTransform.logmel_batch(orig_freq=...))."""
        feats, audio_len = self.transform.logmel_batch(waveform, lengths, ncw_dtype=self.model.storage_dtype,
                                                       orig_freq=self._rate(sample_rate))
        return self.model.greedy(feats, audio_len)

    @torch.no_grad()
    def transcribe_ids(self, waveform: torch.Tensor, lengths: torch.Tensor, blank: int = 0,
                       sample_rate: Optional[int] = None):
        """waveform -> CTC-collapsed token ids on the device: (ids int64 [B, T'] blank-padded, counts int32 [B]).
        `tokenizer.decode(ids[b, :counts[b]])` is then the final text (no merge_repeated pass needed)."""
        tokens, out_len = self(waveform, lengths, sample_rate=sample_rate)
        return K.ctc_collapse(tokens, out_len, blank)

    @torch.no_grad()
    def evaluate(self, waveform: torch.Tensor, lengths: torch.Tensor, text: torch.Tensor, text_len,
                 sample_rate: Optional[int] = None, blank: int = 0):
        """Score a batch against its transcripts, as the reference's validation / test steps do (forward ->
        log_softmax -> nn.CTCLoss(zero_infinity=True), voice100/models/asr.py:105-106,133-152), plus the token errors of
        the greedy transcripts.  text int64 [B, S] padded, text_len [B] (device tensor or host sequence).
        -> (loss fp32 [B] per utterance with zero_infinity, errors int32 [B] = edit distance between the collapsed
        greedy ids and text, ids, counts), where (ids, counts) are exactly what `transcribe_ids` returns.  The batch
        loss the reference logs is `(loss / text_len.clamp_min(1)).mean()`.  v1: log-mel -> encoder -> CTC tail with
        logits -> ctc_loss on those logits in place (log_softmax inside) -> collapse -> edit distance, 33 launches
        and no host synchronisation (capturable when text_len is a device tensor)."""
        feats, audio_len = self.transform.logmel_batch(waveform, lengths, ncw_dtype=self.model.storage_dtype,
                                                       orig_freq=self._rate(sample_rate))
        m = self.model
        logits, tokens, out_len = K.ctc_finalize(m.decoder.run(m.encoder.run(feats)), True, audio_len)
        return self._score(logits.transpose(0, 1), tokens, out_len, text, text_len, blank)

    @staticmethod
    def _score(logits_tbv, tokens, out_len, text, text_len, blank):
        """logits [T', B, V] (a view), greedy tokens int64 [B, T'], valid lengths [B] -> evaluate's four results."""
        loss = K.ctc_loss_batch(logits_tbv, text, out_len, text_len, blank=blank, zero_infinity=True,
                                normalize=True)[0]
        ids, counts = K.ctc_collapse(tokens, out_len, blank)
        return loss, K.edit_distance(ids, counts, text, text_len), ids, counts

    @torch.no_grad()
    def _capture(self, batch: int, samples: int, dev, wav_dtype=torch.float32, sample_rate=None):
        """-> (graph, static waveform, static lengths, static tokens, static out_len) for one fixed shape.  With a
        `sample_rate` the resampled buffer inside the graph is [batch, ceil(n samples / o)]."""
        with torch.cuda.device(dev):
            wav_s = torch.zeros((batch, samples), dtype=wav_dtype, device=dev)
            len_s = torch.full((batch,), samples, dtype=torch.int32, device=dev)
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):          # warm-up outside capture: one-time function attributes, caches
                for _ in range(2):
                    self(wav_s, len_s, sample_rate=sample_rate)
            torch.cuda.current_stream(dev).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                tok_s, out_s = self(wav_s, len_s, sample_rate=sample_rate)
        return graph, wav_s, len_s, tok_s, out_s

    @torch.no_grad()
    def graphed(self, batch: int, samples: int, device="cuda", wav_dtype=torch.float32,
                sample_rate: Optional[int] = None):
        """Capture the whole path (log-mel -> encoder -> head -> argmax: 30 launches, all libv100 kernels) for one
        fixed [batch, samples] shape into a CUDA graph.  Replaying it removes the per-launch gaps: 8-10 % at
        256 x 15 s, 2.5x at 8 x 10 s (which is ~0.3 ms of GPU work behind ~0.7 ms of launches).
        `wav_dtype` torch.float32 or torch.int16 (PCM).  `sample_rate` is the input's rate (None = the transform's);
        another rate adds the resampling kernel to the graph.  Returns `run(waveform, lengths) -> (tokens, out_len)`;
        the outputs are static buffers overwritten by the next replay; `run.graph.replay()` re-runs on the current
        contents of `run.waveform/.lengths`."""
        dev = torch.device(device)
        graph, wav_s, len_s, tok_s, out_s = self._capture(batch, samples, dev, wav_dtype, self._rate(sample_rate))

        def run(waveform: torch.Tensor, lengths: torch.Tensor):
            wav_s.copy_(waveform, non_blocking=True)
            len_s.copy_(lengths, non_blocking=True)
            graph.replay()
            return tok_s, out_s
        run.graph, run.waveform, run.lengths, run.tokens, run.out_len = graph, wav_s, len_s, tok_s, out_s
        return run

    @torch.no_grad()
    def submit_host(self, waveform: torch.Tensor, lengths: torch.Tensor, device="cuda", chunks: int = 4,
                    sample_rate: Optional[int] = None):
        """Asynchronous end-to-end call: host buffers in (pin them for full PCIe speed), host tokens out.
        `waveform` is fp32 or int16 PCM (half the H2D bytes; identical features for 16-bit sources).
        The batch is cut into `chunks` groups of utterances; each group has its own captured CUDA graph with
        static device buffers.  H2D copies run on a side stream straight into those buffers, so chunk i+1
        uploads while chunk i computes, and each chunk's tokens come back with an async D2H.  Returns a
        ticket; `ticket.result()` waits for THIS batch only, so the next batch can be submitted (and start
        uploading) before the previous one has finished computing.  Two tickets may be in flight: consecutive
        calls alternate between two sets of graphs / device buffers, so batch i+1 uploads into its own buffers
        while batch i still computes.  `chunks=1` gives the best throughput (whole-batch kernels, uploads hidden
        behind the previous batch), more chunks give a shorter latency for a single batch.
        `sample_rate` is the input's rate (None = the transform's); another rate is resampled inside each graph, so
        the upload stays at the input's size."""
        dev = torch.device(device)
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        B, L = waveform.shape
        n = max(1, min(chunks, B))
        if getattr(self, "_copy_stream", None) is None or self._copy_stream.device != dev:
            self._copy_stream = torch.cuda.Stream(dev)
            self._host_out, self._slot, self._chunk_graphs = {}, 0, {}
        rate = self._rate(sample_rate)
        L_feat = L if rate is None else resampled_length(L, rate, self.transform.sample_rate)
        T_out = (self.transform.num_frames(L_feat) + 1) // 2
        slot = self._slot
        key = (B, T_out, slot)
        self._slot ^= 1                      # double-buffered device inputs and pinned outputs: two tickets in flight
        if key not in self._host_out:
            self._host_out[key] = (torch.empty((B, T_out), dtype=torch.int64).pin_memory(),
                                   torch.empty((B,), dtype=torch.int32).pin_memory())
        tok_h, len_h = self._host_out[key]
        with torch.cuda.device(dev):
            cur = torch.cuda.current_stream(dev)
            staged = []
            for i in range(n):
                a, b = B * i // n, B * (i + 1) // n
                gkey = (i, b - a, L, slot, waveform.dtype, rate)
                if gkey not in self._chunk_graphs:
                    self._chunk_graphs[gkey] = list(self._capture(b - a, L, dev, waveform.dtype, rate)) + [None]
                cg = self._chunk_graphs[gkey]
                graph, wav_s, len_s, tok_s, out_s, done = cg
                with torch.cuda.stream(self._copy_stream):
                    if done is not None:
                        self._copy_stream.wait_event(done)   # the previous replay has finished reading wav_s
                    wav_s.copy_(waveform[a:b], non_blocking=True)
                    len_s.copy_(lengths[a:b], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(self._copy_stream)
                staged.append((a, b, cg, ev))
            for a, b, cg, ev in staged:
                graph, wav_s, len_s, tok_s, out_s, _ = cg
                cur.wait_event(ev)
                graph.replay()
                tok_h[a:b].copy_(tok_s, non_blocking=True)
                len_h[a:b].copy_(out_s, non_blocking=True)
                cg[5] = torch.cuda.Event()
                cg[5].record(cur)
            done_all = torch.cuda.Event()
            done_all.record(cur)
        return _Ticket(done_all, tok_h, len_h)

    def transcribe_host(self, waveform: torch.Tensor, lengths: torch.Tensor, device="cuda", chunks: int = 4,
                        sample_rate: Optional[int] = None):
        """Synchronous form of submit_host -> (tokens int64 [B, T'] pinned host tensor, valid lengths [B])."""
        return self.submit_host(waveform, lengths, device, chunks, sample_rate).result()


class _Ticket:
    def __init__(self, event, tokens, lengths):
        self._event, self._tokens, self._lengths = event, tokens, lengths

    def result(self):
        self._event.synchronize()
        return self._tokens, self._lengths
