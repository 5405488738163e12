"""Tensor-level wrappers over the C ABI: torch is used for device memory and the current stream only.

All activations are `Ncw` objects: bf16 (or fp32 for head outputs) tensors of shape [B, C, pitch] whose
first `T` columns are data (pitch = T rounded up to 8 so every row starts 16-byte aligned, which is
what TMA and the 16-byte vector accesses in the kernels require).
"""
from __future__ import annotations

from dataclasses import dataclass

import torch

from . import _lib

ACT_NONE, ACT_RELU6 = 0, 1
MEL_LOG_BF16_NCW, MEL_LOG_F32_NTC, MEL_POWER_F32_NCW, MEL_LOG_F16_NCW = 0, 1, 2, 3
DTYPE_CODE = {torch.bfloat16: 0, torch.float16: 1}   # V100_DTYPE_*


def dt(t) -> int:
    """V100_DTYPE_* code of a storage tensor / torch dtype; anything but bf16/fp16 is an error."""
    d = t if isinstance(t, torch.dtype) else t.dtype
    if d not in DTYPE_CODE:
        raise _lib.V100Error(f"storage dtype must be torch.bfloat16 or torch.float16, got {d}")
    return DTYPE_CODE[d]


def _call(anchor, name, *args):
    """Invoke entry point `name` on the device that holds `anchor` (a tensor or Ncw/Tm): the C side launches on
    cudaGetDevice()'s device, so that device is made current for the call and the stream passed is ITS current
    stream -- a model living on cuda:1 works without torch.cuda.set_device(1)."""
    t = anchor if isinstance(anchor, torch.Tensor) else anchor.data
    dev = t.device
    if dev.type != "cuda":
        raise _lib.V100Error("voice100_b200 kernels need CUDA tensors (there is no CPU path)")
    if torch.cuda.current_device() == dev.index:
        return _lib.call(name, *args, torch.cuda.current_stream(dev).cuda_stream)
    with torch.cuda.device(dev):
        return _lib.call(name, *args, torch.cuda.current_stream(dev).cuda_stream)


def _same_device(*tensors):
    """All operands of one call must live on one GPU (a mixed call would hand the kernel a foreign pointer)."""
    devs = {(t if isinstance(t, torch.Tensor) else t.data).device for t in tensors if t is not None}
    if len(devs) > 1:
        raise _lib.V100Error(f"operands of one kernel call live on different devices: {sorted(map(str, devs))}")


def _ptr(t):
    return None if t is None else t.data_ptr()


def pitch_of(T: int, mult: int = 8) -> int:
    return (T + mult - 1) // mult * mult


@dataclass
class Ncw:
    data: torch.Tensor  # [B, C, pitch]
    T: int

    @property
    def B(self):
        return self.data.shape[0]

    @property
    def C(self):
        return self.data.shape[1]

    @property
    def pitch(self):
        return self.data.shape[2]

    def valid(self) -> torch.Tensor:
        return self.data[:, :, : self.T]


def empty_ncw(B, C, T, device, dtype=torch.bfloat16) -> Ncw:
    return Ncw(torch.empty((B, C, pitch_of(T)), device=device, dtype=dtype), T)


def _cuda(t: torch.Tensor, dtype=None):
    if not t.is_cuda:
        raise _lib.V100Error("voice100_b200 kernels need CUDA tensors (there is no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise _lib.V100Error(f"expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise _lib.V100Error("expected a contiguous tensor")
    return t


def logmel(wav: torch.Tensor, lengths: torch.Tensor, fb, log_offset: float, T: int, mode: int, config=None):
    """wav fp32 or int16 PCM [B, L]; lengths int32 [B] (device); fb = (start, count, off, w) device tensors.
    -> (features, audio_len int32 [B] = 1 + len // hop, written by the same kernel).
    `config` = (n_fft, win_length, hop_length, n_mels); None or (512, 400, 160, 64) runs the tuned kernel, anything else
    the generic one (v100_logmel_generic)."""
    nm = 64 if config is None else int(config[3])
    _cuda(lengths, torch.int32)
    if wav.dtype not in (torch.float32, torch.int16):
        raise _lib.V100Error(f"waveforms must be float32 or int16 PCM, got {wav.dtype}")
    _cuda(wav)
    _same_device(wav, lengths, fb[3])
    B = wav.shape[0]
    if mode in (MEL_LOG_BF16_NCW, MEL_LOG_F16_NCW):
        out = empty_ncw(B, nm, T, wav.device, torch.bfloat16 if mode == MEL_LOG_BF16_NCW else torch.float16)
        optr, pitch = out.data.data_ptr(), out.pitch
    elif mode == MEL_POWER_F32_NCW:
        out = Ncw(torch.empty((B, nm, pitch_of(T, 4)), device=wav.device, dtype=torch.float32), T)
        optr, pitch = out.data.data_ptr(), out.pitch
    else:
        out = torch.empty((B, T, nm), device=wav.device, dtype=torch.float32)
        optr, pitch = out.data_ptr(), nm
    frames = torch.empty((B,), device=wav.device, dtype=torch.int32)
    if config is not None and tuple(int(c) for c in config) != (512, 400, 160, 64):
        n_fft, win, hop, _ = (int(c) for c in config)
        _call(wav, "v100_logmel_generic", wav.data_ptr(), 1 if wav.dtype == torch.int16 else 0, lengths.data_ptr(), B,
              wav.stride(0), wav.shape[1], n_fft, win, hop, nm, fb[0].data_ptr(), fb[1].data_ptr(), fb[2].data_ptr(),
              fb[3].data_ptr(), float(log_offset), optr, T, pitch, mode, frames.data_ptr())
        return out, frames
    _call(wav, "v100_logmel", wav.data_ptr(), 1 if wav.dtype == torch.int16 else 0, lengths.data_ptr(), B,
          wav.stride(0), wav.shape[1], fb[0].data_ptr(), fb[1].data_ptr(), fb[2].data_ptr(), fb[3].data_ptr(),
          fb[3].numel(), float(log_offset), optr, T, pitch, mode, frames.data_ptr())
    return out, frames


def ntc_f32_to_ncw(x: torch.Tensor, dtype=torch.bfloat16) -> Ncw:
    _cuda(x, torch.float32)
    B, T, Cc = x.shape
    y = empty_ncw(B, Cc, T, x.device, dtype)
    _call(x, "v100_ntc_f32_to_ncw16", x.data_ptr(), y.data.data_ptr(), B, T, Cc, y.pitch, dt(dtype))
    return y


def ncw_from_f32(x: torch.Tensor, dtype=torch.bfloat16) -> Ncw:
    _cuda(x, torch.float32)
    B, Cc, T = x.shape
    y = empty_ncw(B, Cc, T, x.device, dtype)
    _call(x, "v100_ncw_f32_to_16", x.data_ptr(), y.data.data_ptr(), y.pitch, B, Cc, T, dt(dtype))
    return y


def ncw_to_f32(x: Ncw) -> torch.Tensor:
    y = torch.empty((x.B, x.C, x.T), device=x.data.device, dtype=torch.float32)
    _call(x, "v100_ncw_16_to_f32", x.data.data_ptr(), x.pitch, y.data_ptr(), x.B, x.C, x.T, dt(x.data))
    return y


def conv1x1(x: Ncw, W: torch.Tensor, scale, shift, act: int, res: Ncw = None) -> Ncw:
    C_out, C_in = W.shape
    assert C_in == x.C, (C_in, x.C)
    assert W.dtype == x.data.dtype, "weights and activations must share the storage dtype"
    _same_device(x, W, scale, shift, res)
    y = empty_ncw(x.B, C_out, x.T, x.data.device, x.data.dtype)
    if res is not None:
        assert res.data.shape == y.data.shape and res.T == x.T and res.data.dtype == x.data.dtype
    _call(x, "v100_conv1x1", x.data.data_ptr(), x.pitch, W.data_ptr(), _ptr(scale), shift.data_ptr(),
              None if res is None else res.data.data_ptr(), y.data.data_ptr(), y.pitch, x.B, C_in, C_out, x.T,
              act, dt(x.data))
    return y


def conv1x1_f32(x: Ncw, W: torch.Tensor, bias: torch.Tensor) -> Ncw:
    C_out, C_in = W.shape
    assert C_in == x.C and W.dtype == x.data.dtype
    y = Ncw(torch.empty((x.B, C_out, x.pitch), device=x.data.device, dtype=torch.float32), x.T)
    _call(x, "v100_conv1x1_f32out", x.data.data_ptr(), x.pitch, W.data_ptr(), bias.data_ptr(), y.data.data_ptr(),
              y.pitch, x.B, C_in, C_out, x.T, dt(x.data))
    return y


def dwconv(x: Ncw, w: torch.Tensor, scale, shift, k: int, stride: int, act: int, simt: bool = False) -> Ncw:
    T_out = (x.T - 1) // stride + 1
    assert w.dtype == x.data.dtype
    _same_device(x, w, scale, shift)
    y = empty_ncw(x.B, x.C, T_out, x.data.device, x.data.dtype)
    _call(x, "v100_dwconv1d_simt" if simt else "v100_dwconv1d", x.data.data_ptr(), x.pitch,
              w.data_ptr(), _ptr(scale), shift.data_ptr(), y.data.data_ptr(), y.pitch, x.B, x.C, x.T, k, stride,
              act, dt(x.data))
    return y


def convtranspose_k5s2(x: Ncw, Wp: torch.Tensor, bias: torch.Tensor) -> Ncw:
    C_out = Wp.shape[0]
    assert Wp.shape[1] == 5 * x.C and Wp.dtype == x.data.dtype
    y = empty_ncw(x.B, C_out, 2 * x.T - 1, x.data.device, x.data.dtype)
    ws = torch.empty((x.B, 3 * x.C, x.pitch), device=x.data.device, dtype=x.data.dtype)
    _call(x, "v100_convtranspose1d_k5s2", x.data.data_ptr(), x.pitch, Wp.data_ptr(), bias.data_ptr(),
              ws.data_ptr(), y.data.data_ptr(), y.pitch, x.B, x.C, C_out, x.T, dt(x.data))
    return y


_status_words = {}


def _status_word(device) -> torch.Tensor:
    """One sticky int32 status word per device (V100_STATUS_* bits), shared by the index-consuming kernels."""
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    if key not in _status_words:
        _status_words[key] = torch.zeros((1,), device=device, dtype=torch.int32)
    return _status_words[key]


def embedding_ncw(ids: torch.Tensor, table: torch.Tensor, validate: bool = True) -> Ncw:
    """ids int64 [B, T] -> 16-bit Ncw [B, C, T].  nn.Embedding raises IndexError for an id outside [0, V); with
    `validate` (default) so does this wrapper -- it reads the kernel's sticky status word back, one tiny D2H sync.
    Pass validate=False inside CUDA-graph capture (the column of a bad id is then zero and the flag stays set)."""
    _cuda(ids, torch.int64)
    _same_device(ids, table)
    B, T = ids.shape
    V, Cc = table.shape
    dt(table)
    y = empty_ncw(B, Cc, T, ids.device, table.dtype)
    status = _status_word(ids.device)
    _call(ids, "v100_embedding_ncw16", ids.data_ptr(), table.data_ptr(), y.data.data_ptr(), y.pitch, B, T, V, Cc,
          status.data_ptr())
    if validate and not torch.cuda.is_current_stream_capturing():
        if int(status.item()) & 1:
            status.zero_()
            raise IndexError(f"embedding id outside [0, {V}) (nn.Embedding raises the same IndexError)")
    return y


def ctc_finalize(y: Ncw, want_logits: bool = True, audio_len: torch.Tensor = None):
    """-> (logits [B, T, V] or None, tokens int64 [B, T]) and, when `audio_len` (int32 [B], device) is given, also
    out_len int32 [B] = (audio_len + 1) // 2 written by the same kernel (AudioToTextCTC.output_length)."""
    B, V, T = y.B, y.C, y.T
    logits = torch.empty((B, T, V), device=y.data.device, dtype=torch.float32) if want_logits else None
    tokens = torch.empty((B, T), device=y.data.device, dtype=torch.int64)
    out_len = None
    if audio_len is not None:
        _cuda(audio_len, torch.int32)
        _same_device(y, audio_len)
        out_len = torch.empty((B,), device=y.data.device, dtype=torch.int32)
    _call(y, "v100_ctc_finalize", y.data.data_ptr(), y.pitch, _ptr(logits), tokens.data_ptr(), B, V, T,
          _ptr(audio_len), _ptr(out_len))
    return (logits, tokens) if audio_len is None else (logits, tokens, out_len)


def ctc_collapse(tokens: torch.Tensor, valid_len: torch.Tensor = None, blank: int = 0):
    """tokens int64 [B, T] (+ valid lengths) -> (collapsed ids int64 [B, T] blank-padded, counts int32 [B])."""
    _cuda(tokens, torch.int64)
    B, T = tokens.shape
    out = torch.empty_like(tokens)
    out_len = torch.empty((B,), device=tokens.device, dtype=torch.int32)
    vl = None if valid_len is None else valid_len.to(device=tokens.device, dtype=torch.int64).contiguous()
    _call(tokens, "v100_ctc_collapse", tokens.data_ptr(), _ptr(vl), out.data_ptr(), out_len.data_ptr(), B, T, int(blank))
    return out, out_len


def ctc_best_path(logprob: torch.Tensor, logit_len: torch.Tensor, text: torch.Tensor, text_len: torch.Tensor,
                  normalize: bool = False):
    """logprob fp32 [B, T, V] (raw logits when `normalize`: the kernel applies log_softmax), logit_len [B],
    text int64 [B, L], text_len [B] -> (score fp32 [B], path int32 [B, T] state indices, path_labels int64 [B, T])."""
    _cuda(logprob, torch.float32), _cuda(text, torch.int64)
    _same_device(logprob, text)
    B, T, V = logprob.shape
    L = text.shape[1]
    dev = logprob.device
    ll = logit_len.to(device=dev, dtype=torch.int32).contiguous()
    tl = text_len.to(device=dev, dtype=torch.int32).contiguous()
    ws = torch.empty((B, T, 2 * L + 1), device=dev, dtype=torch.uint8)
    score = torch.empty((B,), device=dev, dtype=torch.float32)
    path = torch.empty((B, T), device=dev, dtype=torch.int32)
    labels = torch.empty((B, T), device=dev, dtype=torch.int64)
    _call(logprob, "v100_ctc_best_path", logprob.data_ptr(), ll.data_ptr(), text.data_ptr(), tl.data_ptr(),
          ws.data_ptr(), score.data_ptr(), path.data_ptr(), labels.data_ptr(), B, T, V, L, 1 if normalize else 0)
    return score, path, labels


def world_finalize(y: Ncw, mean, std, unnormalize: bool, logspc_size: int = 257, codeap_size: int = 1,
                   layout: int = 1):
    """Decoder output Ncw fp32 -> layout 1: (hasf0, f0, logspc, codeap); layout 2: (hasf0, f0, logspc, hascodeap,
    codeap).  See v100_world_finalize."""
    B, T, dev = y.B, y.T, y.data.device
    S, A = logspc_size, codeap_size
    assert y.C == 2 + S + (2 if layout == 2 else 1) * A, (y.C, S, A, layout)
    _same_device(y, mean, std)
    hasf0 = torch.empty((B, T), device=dev, dtype=torch.float32)
    f0 = torch.empty((B, T), device=dev, dtype=torch.float32)
    logspc = torch.empty((B, T, S), device=dev, dtype=torch.float32)
    hascodeap = torch.empty((B, T, A), device=dev, dtype=torch.float32) if layout == 2 else None
    codeap = torch.empty((B, T, A), device=dev, dtype=torch.float32)
    _call(y, "v100_world_finalize", y.data.data_ptr(), y.pitch, _ptr(mean), _ptr(std), hasf0.data_ptr(),
          f0.data_ptr(), logspc.data_ptr(), _ptr(hascodeap), codeap.data_ptr(), B, T, S, A, layout,
          1 if unnormalize else 0)
    return (hasf0, f0, logspc, codeap) if layout == 1 else (hasf0, f0, logspc, hascodeap, codeap)


def ncw_f32_to_ntc(y: Ncw) -> torch.Tensor:
    out = torch.empty((y.B, y.T, y.C), device=y.data.device, dtype=torch.float32)
    _call(y, "v100_ncw_f32_to_ntc", y.data.data_ptr(), y.pitch, out.data_ptr(), y.B, y.C, y.T)
    return out


def maskaudio(audio: torch.Tensor, audio_len: torch.Tensor, log_offset: float) -> torch.Tensor:
    """audio fp32 [B, T, C], audio_len [B] -> log(clamp(exp(audio) * (t < len), min=log_offset)) (voice100/audio.py:106-108)."""
    if audio.dim() != 3 or audio.dtype != torch.float32:
        raise _lib.V100Error("maskaudio: audio must be fp32 [B, T, C]")
    audio = audio.contiguous()
    if audio_len.is_cuda:
        _same_device(audio, audio_len)
    lens = audio_len.to(device=audio.device, dtype=torch.int32).contiguous()
    if lens.shape != (audio.shape[0],):
        raise _lib.V100Error("maskaudio: audio_len must be [B]")
    out = torch.empty_like(audio)
    _call(audio, "v100_maskaudio", audio.data_ptr(), lens.data_ptr(), out.data_ptr(), audio.shape[0], audio.shape[1],
          audio.shape[2], float(log_offset))
    return out


# ---- v2 models: dense conv + LayerNorm/GELU, time-major layout, LSTM (include/v100.h, "v2 models") ----

def conv1d(x: Ncw, Wp: torch.Tensor, bias: torch.Tensor, k: int, stride: int, pad: int) -> Ncw:
    """Dense Conv1d; Wp is the tap-major packed weight [C_out, k*C_in]."""
    C_out = Wp.shape[0]
    assert Wp.shape[1] == k * x.C and Wp.dtype == x.data.dtype
    T_out = (x.T + 2 * pad - k) // stride + 1
    y = empty_ncw(x.B, C_out, T_out, x.data.device, x.data.dtype)
    ws = torch.empty((x.B, k * x.C, y.pitch), device=x.data.device, dtype=x.data.dtype)
    _call(x, "v100_conv1d", x.data.data_ptr(), x.pitch, Wp.data_ptr(), bias.data_ptr(), ws.data_ptr(),
              y.data.data_ptr(), y.pitch, x.B, x.C, C_out, x.T, k, stride, pad, dt(x.data))
    return y


def layernorm_gelu(x: Ncw, gamma: torch.Tensor, beta: torch.Tensor, eps: float) -> Ncw:
    """LayerNorm over channels + GELU(erf), in place."""
    _call(x, "v100_layernorm_gelu", x.data.data_ptr(), x.pitch, gamma.data_ptr(), beta.data_ptr(), float(eps),
              x.data.data_ptr(), x.pitch, x.B, x.C, x.T, dt(x.data))
    return x


@dataclass
class Tm:
    """Time-major activations: data [C, T*Bp] with column t*Bp + b; also a 1-utterance Ncw of T*Bp columns."""
    data: torch.Tensor
    B: int
    T: int
    Bp: int

    @property
    def C(self):
        return self.data.shape[0]

    def as_ncw(self) -> Ncw:
        return Ncw(self.data.view(1, self.data.shape[0], self.data.shape[1]), self.T * self.Bp)


def ncw_to_tm(x: Ncw) -> Tm:
    Bp = pitch_of(x.B)
    y = torch.empty((x.C, x.T * Bp), device=x.data.device, dtype=x.data.dtype)
    _call(x, "v100_ncw_to_tm", x.data.data_ptr(), x.pitch, y.data_ptr(), x.B, x.C, x.T, Bp)
    return Tm(y, x.B, x.T, Bp)


def conv1d_tm(x: Tm, Wp: torch.Tensor, bias: torch.Tensor, k: int) -> Tm:
    """Dense Conv1d, stride 1, padding (k-1)/2, on a time-major tensor; Wp tap-major [C_out, k*C_in]."""
    C_out = Wp.shape[0]
    assert Wp.shape[1] == k * x.C and Wp.dtype == x.data.dtype
    y = torch.empty((C_out, x.T * x.Bp), device=x.data.device, dtype=x.data.dtype)
    _call(x, "v100_conv1d_tm", x.data.data_ptr(), Wp.data_ptr(), bias.data_ptr(), y.data_ptr(), x.C, C_out, x.T,
              x.Bp, k, dt(x.data))
    return Tm(y, x.B, x.T, x.Bp)


def layernorm_gelu_tm(x: Tm, gamma: torch.Tensor, beta: torch.Tensor, eps: float) -> Tm:
    layernorm_gelu(x.as_ncw(), gamma, beta, eps)
    return x


def tm_to_ncw(x: Tm) -> Ncw:
    y = empty_ncw(x.B, x.C, x.T, x.data.device, x.data.dtype)
    _call(x, "v100_tm_to_ncw", x.data.data_ptr(), y.data.data_ptr(), y.pitch, x.B, x.C, x.T, x.Bp)
    return y


# ---- TTS text alignment (v100_tts_align) ----

ALIGN_OK, ALIGN_INDEX, ALIGN_NEGATIVE, ALIGN_NAN, ALIGN_INF, ALIGN_TOO_LONG, ALIGN_CAPACITY = range(7)   # V100_ALIGN_*
ALIGN_FAILED = (ALIGN_INDEX, ALIGN_NEGATIVE, ALIGN_NAN, ALIGN_INF, ALIGN_TOO_LONG)


def tts_align(text: torch.Tensor, align: torch.Tensor, text_len, rule: int, head: int, tail: int, T_cap,
              log1p: bool, durations_out: torch.Tensor = None):
    """One v100_tts_align call.  text int64 [B, L], align fp32 [B, L, 2] with any strides (a strided view of a head
    output is read in place), text_len int32 [B] on the device or None.  T_cap None is a plan-only call.
    -> (aligntext int64 [B, T_cap] or None, int32 [4, B] = aligntext_len, status, filled_len, frame_len)."""
    if text.dtype != torch.int64 or not text.is_cuda or text.dim() != 2:
        raise _lib.V100Error("tts_align: text must be a CUDA int64 [B, L] tensor")
    if text.stride(1) != 1:
        text = text.contiguous()                          # rows may be strided, tokens within a row may not
    if align.dtype != torch.float32 or not align.is_cuda or align.dim() != 3 or align.shape[2] != 2:
        raise _lib.V100Error("tts_align: align must be a CUDA fp32 [B, L, 2] tensor")
    B, L = text.shape
    if tuple(align.shape[:2]) != (B, L):
        raise _lib.V100Error(f"tts_align: align {tuple(align.shape)} does not match text {tuple(text.shape)}")
    if text_len is not None:
        _cuda(text_len, torch.int32)
    if durations_out is not None:
        _cuda(durations_out, torch.float32)
        if tuple(durations_out.shape) != (B, L, 2):
            raise _lib.V100Error(f"tts_align: durations_out must be [{B}, {L}, 2]")
    _same_device(text, align, text_len, durations_out)
    dev = text.device
    at = None if T_cap is None else torch.empty((B, T_cap), device=dev, dtype=torch.int64)
    out = torch.empty((4, B), device=dev, dtype=torch.int32)
    _call(text, "v100_tts_align", align.data_ptr(), align.stride(0), align.stride(1), align.stride(2),
          1 if log1p else 0, _ptr(durations_out), text.data_ptr(), text.stride(0), _ptr(text_len), B, L, rule, head,
          tail, _ptr(at), 0 if T_cap is None else T_cap, out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
          out[3].data_ptr())
    return at, out


def _raise_align_status(code: int, b: int):
    """The exception the host loop raises for the utterance the kernel flagged."""
    where = f"utterance {b}"
    if code == ALIGN_INDEX:
        raise IndexError(f"{where}: a frame index falls outside the aligned text (the reference loop raises here)")
    if code == ALIGN_NEGATIVE:
        raise RuntimeError(f"{where}: Trying to create tensor with negative dimension (the total length is negative)")
    if code == ALIGN_NAN:
        raise ValueError(f"{where}: cannot convert float NaN to integer (the duration sum is NaN)")
    if code == ALIGN_INF:
        raise OverflowError(f"{where}: cannot convert float infinity to integer (the duration sum is infinite)")
    raise _lib.V100Error(f"{where}: the aligned text has 2^31 frames or more")


def align_frames(text: torch.Tensor, align: torch.Tensor, text_len: torch.Tensor = None, rule: int = 1,
                 head: int = 5, tail: int = 5, max_frames: int = None, log1p: bool = False,
                 durations_out: torch.Tensor = None):
    """Per-token (gap, duration) -> aligned text on the device: the batched, bit-exact form of
    TextToAlignTextModel.align (rule=1, tts.py:89-110) and TextToAlignText.align (rule=2, _align_v2.py:54-82).
    text int64 [B, L], align fp32 [B, L, 2] on the device (any strides), text_len [B] (None = all L tokens).
    `log1p=True` applies exp(x) - 1 to `align` first (the head output is log(1 + duration)); `durations_out`, an
    fp32 [B, L, 2] device tensor, then receives the durations.

    Without `max_frames`: a plan call, one device-to-host copy of the lengths and status codes (8 bytes an utterance)
    and an exact-size fill -> (aligntext int64 [B, max total], aligntext_len int32 [B]) on the device.  Where the host
    loop fails, this raises the same exception class for the first such utterance (IndexError, RuntimeError,
    ValueError, OverflowError).

    With `max_frames`: one launch, no host synchronisation, nothing raised (CUDA-graph capturable) ->
    (aligntext int64 [B, max_frames], aligntext_len int32 [B] clamped to max_frames, status int32 [B]).  status is
    ALIGN_OK, one of ALIGN_FAILED (the row is all 0 and its length 0), or ALIGN_CAPACITY (the utterance was cut to
    its first max_frames frames).

    Rule 2 follows the reference loop where align_batch_v2 does not: frames at or past the total length are dropped
    (the slice assignment of TextToAlignText.align), where align_batch_v2 raises IndexError."""
    if rule not in (1, 2):
        raise ValueError(f"rule must be 1 or 2, got {rule}")
    dev = align.device
    text = text.to(dev)
    if text_len is not None:
        text_len = text_len.to(device=dev, dtype=torch.int32).contiguous()
    if max_frames is not None:
        at, out = tts_align(text, align, text_len, rule, head, tail, int(max_frames), log1p, durations_out)
        return at, out[2], out[1]
    at, out = _align_exact(text, align, text_len, rule, head, tail, log1p, durations_out)
    return at, out[0]


def _align_exact(text, align, text_len, rule, head, tail, log1p, durations_out=None):
    """Plan call, one device-to-host copy of (aligntext_len, status), then the fill at the batch's largest total.
    Raises what the host loop raises for the first failing utterance.  -> tts_align's (aligntext, [4, B] lengths)."""
    _, out = tts_align(text, align, text_len, rule, head, tail, None, log1p, durations_out)
    plan = out[:2].cpu()                                  # the one host round trip
    bad = (plan[1] != ALIGN_OK).nonzero()
    if bad.numel():
        b = int(bad[0, 0])
        _raise_align_status(int(plan[1, b]), b)
    return tts_align(text, align, text_len, rule, head, tail, int(plan[0].max()), log1p)


def lstm_workspace(B: int, H: int, device) -> torch.Tensor:
    n = int(_lib.lib().v100_lstm_workspace_bytes(B, H))
    ws = torch.empty((n + 1024,), device=device, dtype=torch.uint8)
    off = (-ws.data_ptr()) % 1024
    return ws[off:off + n]


def lstm_layer(x: Tm, w_ih: torch.Tensor, bias: torch.Tensor, w_hh: torch.Tensor, lengths: torch.Tensor,
               workspace: torch.Tensor = None) -> Tm:
    """One bidirectional layer: w_ih [8H, I] (forward rows first), bias fp32 [8H] = b_ih + b_hh, w_hh [2, 4H, H],
    lengths int32 [B] on the device."""
    H = w_hh.shape[2]
    assert w_ih.shape == (8 * H, x.C) and w_hh.shape == (2, 4 * H, H) and w_ih.dtype == w_hh.dtype == x.data.dtype
    _cuda(lengths, torch.int32)
    gx = conv1x1(x.as_ncw(), w_ih, None, bias, ACT_NONE)           # [1, 8H, T*Bp]: every step's input projection
    y = torch.empty((2 * H, x.T * x.Bp), device=x.data.device, dtype=x.data.dtype)
    ws = workspace if workspace is not None else lstm_workspace(x.B, H, x.data.device)
    _call(x, "v100_lstm_layer", gx.data.data_ptr(), w_hh.data_ptr(), lengths.data_ptr(), y.data_ptr(),
              ws.data_ptr(), x.B, x.Bp, x.T, H, dt(x.data))
    return Tm(y, x.B, x.T, x.Bp)


# ---------------------------------------------------------------------------------------------- WORLD synthesis

WORLD_OK, WORLD_SHORT, WORLD_NONFINITE = 0, 1, 2      # V100_WORLD_*
WORLD_FS, WORLD_FFT, WORLD_HOP, WORLD_BINS = 16000, 512, 160, 257
_WORLD_NOISE_MIN = 1 << 20                            # values (65 s of audio) in the first table of a device
_world_noise = {}                                     # device index -> float64 table (WORLD's randn stream)
_world_noise_retired = []                             # replaced tables stay alive: captured graphs may still read them


def world_noise(n: int, device) -> torch.Tensor:
    """WORLD's randn() stream (v100_world_noise) as a float64 device tensor of at least n values, built once per
    device and grown (to at least twice its size) when a longer one is needed.  Growing launches a kernel and allocates,
    so it must happen outside CUDA-graph capture: a captured call that needs more than the table holds raises."""
    dev = torch.device(device)
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    tab = _world_noise.get(dev.index)
    if tab is None or tab.numel() < n:
        if torch.cuda.is_current_stream_capturing():
            raise _lib.V100Error(f"the WORLD noise table holds {0 if tab is None else tab.numel()} values and {n} are "
                                 "needed: run the call once before graph capture so that the table is built there")
        m = max(int(n), _WORLD_NOISE_MIN, 2 * (0 if tab is None else tab.numel()))
        new = torch.empty((m,), device=dev, dtype=torch.float64)
        _call(new, "v100_world_noise", new.data_ptr(), m)
        if tab is not None:
            _world_noise_retired.append(tab)
        _world_noise[dev.index] = tab = new
    return tab


def _world_inputs(f0, logspc, codeap, frame_len):
    if f0.dim() != 2 or logspc.dim() != 3:
        raise _lib.V100Error(f"WORLD synthesis: f0 must be [B, T] and logspc [B, T, {WORLD_BINS}]")
    if codeap.dim() == 2:
        codeap = codeap.unsqueeze(-1)
    B, T = f0.shape
    if logspc.shape[2] != WORLD_BINS:
        raise _lib.V100Error(f"WORLD synthesis: logspc has {logspc.shape[2]} bins; the 16 kHz / 512-point vocoder "
                             f"needs {WORLD_BINS} (25 mel-cepstra: decode them with AlignTextToAudioPredict)")
    if codeap.dim() != 3 or codeap.shape[2] != 1:
        raise _lib.V100Error(f"WORLD synthesis: codeap must be [B, T, 1] (one band at 16 kHz), got {tuple(codeap.shape)}")
    if tuple(logspc.shape[:2]) != (B, T) or tuple(codeap.shape[:2]) != (B, T):
        raise _lib.V100Error(f"WORLD synthesis: shapes f0 {tuple(f0.shape)}, logspc {tuple(logspc.shape)}, codeap "
                             f"{tuple(codeap.shape)} do not agree")
    for t in (f0, logspc, codeap):
        if t.dtype != torch.float32 or not t.is_cuda:
            raise _lib.V100Error("WORLD synthesis: f0, logspc and codeap must be fp32 CUDA tensors")
    if frame_len is not None:
        _cuda(frame_len, torch.int32)
        if tuple(frame_len.shape) != (B,):
            raise _lib.V100Error(f"WORLD synthesis: frame_len must be int32 [{B}]")
    _same_device(f0, logspc, codeap, frame_len)
    if B <= 0:
        raise _lib.V100Error("WORLD synthesis: empty batch")
    return B, T, codeap


def _world_workspace(B: int, T: int, device) -> torch.Tensor:
    n = int(_lib.lib().v100_world_workspace_bytes(B, WORLD_HOP * T))
    ws = torch.empty((n + 256,), device=device, dtype=torch.uint8)
    off = (-ws.data_ptr()) % 256
    return ws[off:off + n]


def _world_args(f0, logspc, codeap, frame_len):
    return (f0.data_ptr(), f0.stride(0), f0.stride(1), logspc.data_ptr(), logspc.stride(0), logspc.stride(1),
            logspc.stride(2), codeap.data_ptr(), codeap.stride(0), codeap.stride(1), _ptr(frame_len))


def world_timebase(f0: torch.Tensor, logspc: torch.Tensor, codeap: torch.Tensor, frame_len: torch.Tensor = None):
    """v100_world_timebase alone, decoded for inspection: -> (workspace views) dict with
    head int32 [B, 4] (status, y_len, first pulse, pulse count), info int32 [B, 160 T] (-1, or noise size << 1 | vuv),
    tau float64 [B, 160 T], wav_len int32 [B], status int32 [B]."""
    B, T, codeap = _world_inputs(f0, logspc, codeap, frame_len)
    Yp = (WORLD_HOP * T + 31) // 32 * 32
    ws = _world_workspace(B, T, f0.device)
    out = torch.empty((2, B), device=f0.device, dtype=torch.int32)
    _call(f0, "v100_world_timebase", *_world_args(f0, logspc, codeap, frame_len), B, T, ws.data_ptr(),
          out[0].data_ptr(), out[1].data_ptr())
    a = lambda x: (x + 255) // 256 * 256
    o1, o2 = a(B * 16), a(B * 16) + a(B * Yp * 4)
    return dict(head=ws[:B * 16].view(torch.int32).view(B, 4), info=ws[o1:o1 + B * Yp * 4].view(torch.int32).view(B, Yp),
                tau=ws[o2:o2 + B * Yp * 8].view(torch.float64).view(B, Yp), wav_len=out[0], status=out[1])


def world_synthesize(f0: torch.Tensor, logspc: torch.Tensor, codeap: torch.Tensor, frame_len: torch.Tensor = None,
                     max_samples: int = None):
    """WORLD vocoder on the device (v100_world_synthesize): DecodeAperiodicity + Synthesis at 16 kHz, 512-point FFT,
    10 ms frames, for a padded batch.  f0 fp32 [B, T] (Hz, 0 = unvoiced), logspc fp32 [B, T, 257], codeap fp32 [B, T, 1]
    or [B, T], any strides (read in place); frame_len int32 [B] valid frames (None = T).
    -> (wav fp32 [B, Y], wav_len int32 [B] = 160 frame_len, status int32 [B] = WORLD_*), Y = max_samples (>= 160 T,
    default 160 T).  Samples from wav_len on are 0; a rejected utterance (WORLD_SHORT: fewer than two frames,
    WORLD_NONFINITE: NaN / inf among its parameters) is all 0 with wav_len 0.  No host synchronisation; capturable once
    the noise table of this device is large enough (see world_noise)."""
    B, T, codeap = _world_inputs(f0, logspc, codeap, frame_len)
    Y = WORLD_HOP * T if max_samples is None else int(max_samples)
    if Y < WORLD_HOP * T or Y <= 0:
        raise _lib.V100Error(f"world_synthesize: max_samples = {Y} must be positive and at least 160 T = "
                             f"{WORLD_HOP * T}")
    dev = f0.device
    noise = world_noise(WORLD_HOP * T, dev)
    ws = _world_workspace(B, T, dev)
    wav = torch.empty((B, Y), device=dev, dtype=torch.float32)
    out = torch.empty((2, B), device=dev, dtype=torch.int32)
    _call(f0, "v100_world_synthesize", *_world_args(f0, logspc, codeap, frame_len), B, T, noise.data_ptr(),
          noise.numel(), ws.data_ptr(), wav.data_ptr(), Y, out[0].data_ptr(), out[1].data_ptr())
    return wav, out[0], out[1]


# ---------------------------------------------------------------------------------------------- WORLD analysis

_WORLD_ANALYSIS_DRAWS = 5290                          # dither values a frame can read (LoveTrain + D4C), per frame
_dio_taps = {}                                        # device index -> float64 DIO filter table


def dio_taps(device) -> torch.Tensor:
    """DIO's filters as v100_world_analyze reads them (float64 [1633]): the 641-tap low-cut filter, then the Nuttall
    windows of the 7 bands.  Built with numpy, by the same expressions as oracle/world_analysis.py's dio_taps(), once
    per device and outside graph capture."""
    import numpy as np
    dev = torch.device(device)
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    tab = _dio_taps.get(dev.index)
    if tab is None:
        if torch.cuda.is_current_stream_capturing():
            raise _lib.V100Error("the DIO filter table is built on first use: run world_analyze once before capture")
        pi = 3.1415926535897932384
        i = np.arange(1, 642, dtype=np.float64)
        w = 0.5 - 0.5 * np.cos(i * 2.0 * pi / 642)
        s = 0.0
        for v in w:
            s += v
        low = -w / s
        low[320] += 1.0
        parts = [low]
        for k in range(7):
            x = 16000 / (71.0 * 2.0 ** ((k + 1) / 2.0)) / 2.0
            n = 4 * int(x + 0.5)
            u = np.arange(n, dtype=np.float64) / (n - 1.0)
            parts.append(0.355768 - 0.487396 * np.cos(2.0 * pi * u) + 0.144232 * np.cos(4.0 * pi * u)
                         - 0.012604 * np.cos(6.0 * pi * u))
        tab = torch.from_numpy(np.concatenate(parts)).to(dev)
        _dio_taps[dev.index] = tab
    return tab


def world_analyze(wav: torch.Tensor, lengths: torch.Tensor, T: int = None):
    """WORLD analysis on the device (v100_world_analyze): Dio + StoneMask + CheapTrick + D4C + CodeAperiodicity at
    16 kHz, 10 ms frames, fft_size 512, for a padded batch.  wav fp32 or int16 PCM [B, L] with unit stride along time
    and any row pitch; lengths int32 [B] on the device.
    -> (f0 fp32 [B, T], logspc fp32 [B, T, 257], codeap fp32 [B, T, 1], frame_len int32 [B] = lengths // 160 + 1,
    status int32 [B] = WORLD_*), T = L // 160 + 1 by default.  Rows at and past frame_len are 0; a rejected utterance
    (WORLD_SHORT: fewer than 480 samples, WORLD_NONFINITE: a NaN or inf sample) is all 0 with frame_len 0.  No host
    synchronisation; capturable once this device's noise and filter tables exist (a first call builds them)."""
    _cuda(lengths, torch.int32)
    if wav.dtype not in (torch.float32, torch.int16):
        raise _lib.V100Error(f"world_analyze: waveforms must be float32 or int16 PCM, got {wav.dtype}")
    if not wav.is_cuda or wav.dim() != 2 or wav.stride(1) != 1:
        raise _lib.V100Error("world_analyze: wav must be a CUDA [B, L] tensor with unit stride along time")
    B, L = wav.shape
    if tuple(lengths.shape) != (B,):
        raise _lib.V100Error(f"world_analyze: lengths must be int32 [{B}]")
    _same_device(wav, lengths)
    if B <= 0:
        raise _lib.V100Error("world_analyze: empty batch")
    T = L // WORLD_HOP + 1 if T is None else int(T)
    if T < L // WORLD_HOP + 1:
        raise _lib.V100Error(f"world_analyze: T = {T} frames < L // 160 + 1 = {L // WORLD_HOP + 1}")
    dev = wav.device
    noise = world_noise(_WORLD_ANALYSIS_DRAWS * (L // WORLD_HOP + 1), dev)
    taps = dio_taps(dev)
    n = int(_lib.lib().v100_world_analysis_workspace_bytes(B, L))
    ws = torch.empty((n + 256,), device=dev, dtype=torch.uint8)
    off = (-ws.data_ptr()) % 256
    f0 = torch.empty((B, T), device=dev, dtype=torch.float32)
    logspc = torch.empty((B, T, WORLD_BINS), device=dev, dtype=torch.float32)
    codeap = torch.empty((B, T, 1), device=dev, dtype=torch.float32)
    out = torch.empty((2, B), device=dev, dtype=torch.int32)
    pitch = wav.stride(0) if B > 1 else L
    _call(wav, "v100_world_analyze", wav.data_ptr(), 1 if wav.dtype == torch.int16 else 0, pitch, lengths.data_ptr(),
          B, L, taps.data_ptr(), noise.data_ptr(), noise.numel(), ws.data_ptr() + off, T, f0.data_ptr(),
          logspc.data_ptr(), codeap.data_ptr(), out[0].data_ptr(), out[1].data_ptr())
    return f0, logspc, codeap, out[0], out[1]


# ---------------------------------------------------------------------------------------------- resampling


def resample(wav: torch.Tensor, lengths: torch.Tensor, table, L_out: int):
    """One v100_resample call.  wav fp32 or int16 PCM [B, L] with unit stride along time and any row pitch; lengths
    int32 [B] on the device; table a data_modules.ResampleTable on the same device.
    -> (out fp32 [B, L_out], out_len int32 [B] = min(ceil(n lengths / o), L_out)); no host synchronisation."""
    _cuda(lengths, torch.int32)
    if wav.dtype not in (torch.float32, torch.int16):
        raise _lib.V100Error(f"waveforms must be float32 or int16 PCM, got {wav.dtype}")
    if not wav.is_cuda or wav.dim() != 2 or wav.stride(1) != 1:
        raise _lib.V100Error("resample: wav must be a CUDA [B, L] tensor with unit stride along time")
    _same_device(wav, lengths, table.taps)
    B, L = wav.shape
    pitch = wav.stride(0) if B > 1 else L
    out = torch.empty((B, L_out), device=wav.device, dtype=torch.float32)
    out_len = torch.empty((B,), device=wav.device, dtype=torch.int32)
    if B == 0:
        return out, out_len
    _call(wav, "v100_resample", wav.data_ptr(), 1 if wav.dtype == torch.int16 else 0, lengths.data_ptr(), B, pitch, L,
          table.start.data_ptr(), table.count.data_ptr(), table.off.data_ptr(), _ptr(table.taps), table.taps.numel(),
          table.o, table.n, table.width, out.data_ptr(), L_out, L_out, out_len.data_ptr())
    return out, out_len


# ---------------------------------------------------------------------------------------------- ASR evaluation

CTC_OK, CTC_BAD_LABEL, CTC_BAD_LENGTH = 0, 1, 2       # V100_CTC_*
CTC_MAX_TARGET = 4096                                 # V100_CTC_MAX_TARGET
EDIT_MAX_LEN = 16384                                  # V100_EDIT_MAX_LEN


def _host_lengths(x):
    """Host-resident lengths (list, tuple, CPU tensor) as a Python list; None for a device tensor."""
    if isinstance(x, torch.Tensor) and x.is_cuda:
        return None
    return [int(v) for v in (x.tolist() if isinstance(x, torch.Tensor) else x)]


def _lengths_i32(x, device, what: str, B: int):
    """Lengths as a device int32 [B] tensor.  Device values are not read back: they are clamped into the int32 range,
    so that an out-of-range value stays out of range for the kernel's own check."""
    vals = _host_lengths(x)
    if vals is None:
        if x.device != device:
            raise _lib.V100Error(f"{what} lives on {x.device}, the other operands on {device}")
        if x.shape != (B,):
            raise _lib.V100Error(f"{what} must have shape [{B}], got {tuple(x.shape)}")
        return (x if x.dtype == torch.int32 else x.clamp(-1, 2 ** 31 - 1).to(torch.int32)).contiguous()
    if len(vals) != B:
        raise RuntimeError(f"{what} must be of size batch_size = {B}, got {len(vals)}")
    return torch.tensor([min(max(v, -1), 2 ** 31 - 1) for v in vals], dtype=torch.int32).to(device)


def ctc_loss_batch(log_probs: torch.Tensor, targets: torch.Tensor, input_lengths, target_lengths, blank: int = 0,
                   zero_infinity: bool = False, normalize: bool = False):
    """One v100_ctc_loss call -> (loss fp32 [N], status int32 [N] = CTC_*, target lengths int32 [N] on the device).
    log_probs fp32 [T, N, C] on the device with unit stride along C (any other strides are read in place); targets
    int64 [N, S] (padded) or 1-D (concatenated); lengths as torch accepts them.  Host-resident lengths are checked
    before anything else, raising RuntimeError where torch does; device-resident ones are checked by the kernel (NaN
    and CTC_BAD_LENGTH)."""
    if not isinstance(log_probs, torch.Tensor) or log_probs.dtype != torch.float32 or log_probs.dim() != 3:
        raise _lib.V100Error("ctc_loss: log_probs must be an fp32 [T, N, C] tensor")
    T, B, V = log_probs.shape
    if B == 0 or T == 0:
        raise _lib.V100Error("ctc_loss: empty batch")
    if not 0 <= blank < V:
        raise RuntimeError("blank must be in label range")
    if not isinstance(targets, torch.Tensor) or targets.dim() not in (1, 2) or targets.is_floating_point():
        raise RuntimeError("ctc_loss: targets must be an integer tensor [N, S] or 1-D")
    il_host, tl_host = _host_lengths(input_lengths), _host_lengths(target_lengths)
    for what, vals in (("input_lengths", il_host), ("target_lengths", tl_host)):
        if vals is not None and len(vals) != B:
            raise RuntimeError(f"{what} must be of size batch_size = {B}, got {len(vals)}")
        if vals is not None and min(vals) < 0:
            raise RuntimeError(f"Expected {what} to have value at least 0, but got value {min(vals)}")
    if il_host is not None and max(il_host) > T:
        raise RuntimeError(f"Expected input_lengths to have value at most {T}, but got value {max(il_host)}")
    if targets.dim() == 2:
        if targets.shape[0] != B:
            raise RuntimeError(f"ctc_loss: targets has {targets.shape[0]} rows for a batch of {B}")
        if tl_host is not None and max(tl_host) > targets.shape[1]:
            raise RuntimeError(f"Expected tensor to have size at least {max(tl_host)} at dimension 1, but got size "
                               f"{targets.shape[1]} for argument #2 'targets'")
    elif tl_host is not None and sum(tl_host) > targets.numel():
        raise RuntimeError(f"Expected tensor to have size at least {sum(tl_host)} at dimension 0, but got size "
                           f"{targets.numel()} for argument #2 'targets'")
    if not log_probs.is_cuda:
        raise _lib.V100Error("ctc_loss: voice100_b200 kernels need CUDA tensors (there is no CPU path)")
    if log_probs.stride(2) != 1 and V > 1:
        raise _lib.V100Error("ctc_loss: log_probs needs unit stride along C")
    dev = log_probs.device
    targets = targets.to(device=dev, dtype=torch.int64)
    il = _lengths_i32(input_lengths, dev, "input_lengths", B)
    tl = _lengths_i32(target_lengths, dev, "target_lengths", B)
    off = None
    if targets.dim() == 2:
        if targets.shape[1] > 0 and targets.stride(1) != 1:
            targets = targets.contiguous()
        stride, L_max = targets.stride(0), targets.shape[1]
        numel = (B - 1) * stride + targets.shape[1] if targets.shape[1] else 0
        if tl_host is not None:
            L_max = max(tl_host)                          # known lengths: a wide padded buffer is not a limit
    else:
        targets = targets.contiguous()
        stride, numel = 0, targets.numel()
        if tl_host is not None:
            L_max = max(tl_host)
            off = torch.tensor([sum(tl_host[:b]) for b in range(B)], dtype=torch.int64).to(dev)
        else:
            L_max = min(numel, CTC_MAX_TARGET)
            t64 = tl.to(torch.int64)
            off = (torch.cumsum(t64, 0) - t64).contiguous()
    loss = torch.empty((B,), device=dev, dtype=torch.float32)
    status = torch.empty((B,), device=dev, dtype=torch.int32)
    _call(log_probs, "v100_ctc_loss", log_probs.data_ptr(), log_probs.stride(0), log_probs.stride(1), T, B, V,
          il.data_ptr(), targets.data_ptr() if targets.numel() else None, stride, _ptr(off), numel, tl.data_ptr(),
          int(L_max), int(blank), 1 if normalize else 0, 1 if zero_infinity else 0, loss.data_ptr(),
          status.data_ptr())
    return loss, status, tl


def ctc_loss(log_probs: torch.Tensor, targets: torch.Tensor, input_lengths, target_lengths, blank: int = 0,
             reduction: str = "mean", zero_infinity: bool = False, normalize: bool = False) -> torch.Tensor:
    """torch.nn.functional.ctc_loss on the device (v100_ctc_loss): the forward algorithm in float64, the result in fp32.
    Same signature, layout ([T, N, C] log-probabilities, any strides with unit stride along C) and results as torch's
    CPU kernel; `normalize=True` takes raw logits and applies log_softmax in the kernel (float64), so the logits of the
    ASR heads are read in place.  reduction "none" -> fp32 [N]; "mean" -> (loss / target_lengths.clamp_min(1)).mean();
    "sum" -> loss.sum() (torch's own expressions on the per-utterance vector).  A target label outside [0, C) or a
    device-resident length out of range gives NaN for that utterance; host-resident lengths out of range raise
    RuntimeError before launch, as torch does.  No backward: this is for evaluation."""
    if reduction not in ("none", "mean", "sum"):
        raise ValueError(f"{reduction} is not a valid value for reduction")
    loss, _, tl = ctc_loss_batch(log_probs, targets, input_lengths, target_lengths, blank, zero_infinity, normalize)
    if reduction == "none":
        return loss
    if reduction == "sum":
        return loss.sum()
    return (loss / tl.to(loss.dtype).clamp_min(1)).mean()


def edit_distance(hyp: torch.Tensor, hyp_len, ref: torch.Tensor, ref_len) -> torch.Tensor:
    """Levenshtein distance with unit costs between int64 id sequences on the device (v100_edit_distance).
    hyp int64 [B, Lh], ref int64 [B, Lr] (row strides free, unit stride along the row), hyp_len / ref_len [B] (device
    tensors, host sequences or None = the full width; clamped to [0, width] as ctc_collapse does) -> int32 [B].
    Any int64 is a valid id, so word errors are this function on word ids mapped on the host."""
    for name, t in (("hyp", hyp), ("ref", ref)):
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise _lib.V100Error(f"edit_distance: {name} must be a CUDA tensor (there is no CPU path)")
        if t.dtype != torch.int64 or t.dim() != 2:
            raise _lib.V100Error(f"edit_distance: {name} must be int64 [B, L], got {t.dtype} {tuple(t.shape)}")
    _same_device(hyp, ref)
    B = hyp.shape[0]
    if ref.shape[0] != B or B == 0:
        raise _lib.V100Error(f"edit_distance: batch sizes {B} and {ref.shape[0]} differ or are 0")
    if hyp.shape[1] > EDIT_MAX_LEN or ref.shape[1] > EDIT_MAX_LEN:
        raise _lib.V100Error(f"edit_distance: widths {hyp.shape[1]} / {ref.shape[1]} exceed {EDIT_MAX_LEN}")
    hyp = hyp if hyp.shape[1] == 0 or hyp.stride(1) == 1 else hyp.contiguous()
    ref = ref if ref.shape[1] == 0 or ref.stride(1) == 1 else ref.contiguous()
    dev = hyp.device
    hl = None if hyp_len is None else _lengths_i32(hyp_len, dev, "hyp_len", B)
    rl = None if ref_len is None else _lengths_i32(ref_len, dev, "ref_len", B)
    dist = torch.empty((B,), device=dev, dtype=torch.int32)
    _call(hyp, "v100_edit_distance", hyp.data_ptr() if hyp.numel() else None, hyp.stride(0), _ptr(hl), hyp.shape[1],
          ref.data_ptr() if ref.numel() else None, ref.stride(0), _ptr(rl), ref.shape[1], B, dist.data_ptr())
    return dist
