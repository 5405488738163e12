#!/usr/bin/env python
"""Benchmark of the Voice100 ASR hot path: log-mel + ConvVoiceEncoder + CTC head + greedy argmax.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): ASR audio-seconds per second on `asr_en_base` (AudioToTextCTC(64,512,29,512)),
256 utterances x 15 s of synthetic 16 kHz audio PER GPU (weak scaling: utterances are independent, so
ranks share nothing on the data path; NCCL only reduces the timings).  One step = one pass of the whole
path over one batch.  Prints ONE JSON line on rank 0.

  value     device-resident inputs, CUDA-event timed, max over ranks.
  e2e       same metric through AsrPipeline.submit_host/.result(): pinned HOST waveforms in, HOST tokens out,
            every batch's H2D/D2H inside the timed region (whole-batch CUDA graphs on two alternating sets of
            device buffers: batch i+1 uploads while batch i computes).
  roofline  the dominant kernel (tcgen05 conv GEMM) against the measured bf16 peak; `roofline_all`
            lists every kernel class (depthwise and log-mel against the measured HBM copy bandwidth).
  cpu_baseline / --impl reference
            the CPU oracle (oracle/v100_oracle.py: the reference's arithmetic on torch CPU fp32, all host
            threads) on a bounded sample of the same workload.  The reference project is not part of this
            repository; the oracle is pinned to its outputs by tests/golden.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SAMPLE_RATE = 16000
CLIP_SECONDS = 15
BATCH_PER_GPU = 256
MODEL = dict(audio_size=64, embed_size=512, vocab_size=29, hidden_size=512)
WORKLOAD = "asr_en_base: AudioToTextCTC(64,512,29,512), 256 x 15 s synthetic 16 kHz audio per GPU"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sustained=p["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, arrays):
    """--dump-outputs: write what the timed path returned in its last step as <directory>/<name>.npy, floating point
    as float32 and integers as float64 (exact), so that two builds can be compared output for output.  Every array is
    batch-major; above DUMP_LIMIT_BYTES in all, the same seeded sample of utterances is kept from every array and
    their batch indices are written as sample_rows.npy."""
    import numpy as np
    host = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        host[name] = a.astype(np.float32 if np.issubdtype(a.dtype, np.floating) else np.float64)
    B = {a.shape[0] for a in host.values()}
    assert len(B) == 1, {k: a.shape for k, a in host.items()}
    B = B.pop()
    total = sum(a.nbytes for a in host.values())
    os.makedirs(directory, exist_ok=True)
    if total > DUMP_LIMIT_BYTES:
        keep = max(1, B * (DUMP_LIMIT_BYTES - 8 * B) // total)
        rows = np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
        host = {k: a[rows] for k, a in host.items()}
        np.save(os.path.join(directory, "sample_rows.npy"), rows.astype(np.float64))
    for name, a in host.items():
        np.save(os.path.join(directory, name + ".npy"), a)


# --------------------------------------------------------------------------------------------------
# algorithmic work per launch (SURVEY.md section 8d / DESIGN.md): bf16 activations = 2 B
# --------------------------------------------------------------------------------------------------
def asr_work_model(B, T_in, hidden, embed, vocab, audio_size=64, fused=True):
    """-> list of dicts (kind, flops, bytes) in launch order for one step.  With `fused`, the stride-1 blocks run
    expand + depthwise as one kernel ("expand_dw": the 4x-wide tensor between them is neither written nor read)."""
    from voice100_b200.synth import asr_encoder_blocks
    L = (T_in - 1) * 160  # samples per clip (frames = 1 + L//160)
    work = [dict(kind="logmel", flops=0.0, bytes=4.0 * B * L + 2.0 * 64 * B * T_in)]
    T = T_in
    for ci, co, k, s, res in asr_encoder_blocks(audio_size, embed, hidden):
        h = 4 * ci
        M = B * T
        T_out = (T - 1) // s + 1
        Mo = B * T_out
        if fused and s == 1 and h % 256 == 0:
            work.append(dict(kind="expand_dw", flops=2.0 * M * ci * h + 2.0 * k * h * Mo,
                             bytes=2.0 * M * ci + 2.0 * Mo * h + 2.0 * ci * h + 4.0 * 128 * h))
        else:
            work.append(dict(kind="gemm", flops=2.0 * M * ci * h, bytes=2.0 * M * (ci + h) + 2.0 * ci * h))
            work.append(dict(kind="dwconv", flops=2.0 * k * h * Mo, bytes=2.0 * h * (M + Mo) + 2.0 * h * k))
        work.append(dict(kind="gemm", flops=2.0 * Mo * h * co,
                         bytes=2.0 * Mo * (h + co) + (2.0 * Mo * co if res else 0.0) + 2.0 * h * co))
        T = T_out
    M = B * T
    work.append(dict(kind="gemm", flops=2.0 * M * embed * vocab, bytes=2.0 * M * embed + 4.0 * M * vocab))
    work.append(dict(kind="ctc_finalize", flops=0.0, bytes=4.0 * M * vocab + 8.0 * M))
    return work


class ClockSampler:
    """Samples SM clock + throttle reasons of one GPU every 5 ms through NVML while the timed region runs
    (nvidia-smi -lms cannot start fast enough for a sub-second region; it is the fallback)."""
    BITS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index):
        self.index, self.samples, self.reasons, self._stop, self.thread = index, [], set(), False, None
        self.sm_max = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self._stop:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for name, bit in self.BITS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nv is not None:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()

    def stop(self):
        if self.nv is None:
            try:
                q = "clocks.sm,clocks.max.sm,clocks_event_reasons.active"
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True).stdout
                f = [x.strip() for x in out.strip().split(",")]
                return dict(sm_mhz=float(f[0]), sm_max_mhz=float(f[1]), reasons=["nvml unavailable; single nvidia-smi sample after the run: " + f[2]])
            except Exception:
                return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no clock source available"])
        self._stop = True
        self.thread.join()
        sm = sorted(self.samples)
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=self.sm_max, reasons=sorted(self.reasons),
                    samples=len(sm))


CPU_SAMPLE_CLIPS = 32    # clips per CPU pass: enough rows for 16-32 host threads on the narrow layers


def _cpu_pass_factory(batch):
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import v100_oracle as orc
    from voice100_b200 import synth
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    sd = orc.to_torch_sd(synth.asr_state_dict(**MODEL, seed=1234))
    L = SAMPLE_RATE * CLIP_SECONDS
    wav = torch.from_numpy(synth.noise_waveform(batch, L, seed=1234))

    def one_pass():
        with torch.no_grad():
            audio, _ = orc.logmel_batch(wav, [L] * batch)
            return orc.ctc_greedy(orc.asr_forward(audio, sd))
    return one_pass, torch.get_num_threads()


def cpu_oracle_throughput(min_seconds=10.0, batch=CPU_SAMPLE_CLIPS, max_reps=60):
    """The CPU oracle on a bounded sample of the workload: `batch` x 15 s clips per pass, repeated until
    `min_seconds` of CPU work has been timed.  -> (audio_s_per_s, threads, sample description)."""
    one_pass, threads = _cpu_pass_factory(batch)
    one_pass()  # warm-up
    t_total, reps = 0.0, 0
    while t_total < min_seconds and reps < max_reps:
        t0 = time.perf_counter()
        one_pass()
        t_total += time.perf_counter() - t0
        reps += 1
    value = reps * batch * CLIP_SECONDS / t_total
    return value, threads, f"{reps} passes of {batch} x {CLIP_SECONDS} s clips ({t_total:.1f} s of CPU work)"


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port), all host threads.
    Each step is a bounded sample of the workload (32 of the 256 clips); under torchrun only rank 0 works."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    batch = CPU_SAMPLE_CLIPS
    step, threads = _cpu_pass_factory(batch)
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    steps = max(1, args.steps)
    t0 = time.perf_counter()
    for _ in range(steps):
        tokens = step()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"tokens": tokens})
    value = steps * batch * CLIP_SECONDS / dt
    sample = f"each step = {batch} x {CLIP_SECONDS} s clips of the 256-clip workload on {threads} host threads"
    print(json.dumps({
        "impl": "reference", "metric": "asr_audio_seconds_per_second", "value": value, "unit": "audio-s/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": threads, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def gpu_eager_baseline(dev, batch, steps=3):
    """The same path as stock PyTorch eager ON THIS GPU (cuFFT / cuBLAS / cuDNN through ATen): the oracle's functions
    with tensors on the device, fp32 and bf16 (weights and activations cast wholesale, what `model.to(bfloat16)` does
    to the reference).  A reported comparison point (BASELINE.md section 1 (ii)); libraries never enter the product
    path.  -> dict."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import v100_oracle as orc
    from voice100_b200 import synth
    L = SAMPLE_RATE * CLIP_SECONDS
    out = {"clips": batch, "steps": steps, "what": "torch eager on the same B200: torch.stft + matmul + log, F.conv1d / "
           "F.batch_norm / hardtanh per layer (cuFFT, cuBLAS, cuDNN), argmax"}
    sd32 = {k: v.to(dev) for k, v in orc.to_torch_sd(synth.asr_state_dict(**MODEL, seed=1234)).items()}
    g = torch.Generator(device=dev).manual_seed(99)
    wav = 0.1 * torch.randn((batch, L), device=dev, generator=g)
    for name, dtype in (("f32", torch.float32), ("bf16", torch.bfloat16)):
        sd = sd32 if dtype == torch.float32 else {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in sd32.items()}

        def step():
            with torch.no_grad():
                audio = torch.log(orc.mel_power(wav).transpose(-1, -2) + orc.LOG_OFFSET).to(dtype)
                return orc.ctc_greedy(orc.asr_forward(audio, sd))
        try:
            for _ in range(2):
                step()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1) / steps
            out[name] = {"ms_per_step": round(ms, 3), "value": round(batch * CLIP_SECONDS / (ms * 1e-3), 1), "unit": "audio-s/s"}
        except Exception as exc:  # noqa: BLE001 -- a baseline that cannot run must not take the benchmark down
            out[name] = {"error": f"{type(exc).__name__}: {exc}"[:200]}
        torch.cuda.empty_cache()
    return out


def _graph_leg(torch, dev, fn, W, K, ms_eager):
    """Capture `fn` (fixed shapes, device-resident inputs) into a CUDA graph and time K replays; falls back to the
    eager number if the capture is refused.  -> (ms per step, launch description)"""
    try:
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                fn()
        torch.cuda.current_stream(dev).wait_stream(side)
        for _ in range(W):
            graph.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            graph.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / K, "CUDA graph replay"
    except Exception as exc:
        torch.cuda.synchronize()
        return ms_eager, f"eager (graph capture failed: {type(exc).__name__})"


def run_tts(args):
    """Secondary workload (BASELINE.json configs[2], tts_en_base): text [B,100] -> TextToAlignTextModel ->
    host align_batch (seeded synthetic alignment, SURVEY 8a a11) -> AlignTextToAudioModel.predict -> WORLD
    parameters.  Metric: seconds of output audio (10 ms frames) per second.  Not the headline metric."""
    import numpy as np
    import torch
    import voice100_b200 as v
    from voice100_b200 import _lib, synth
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    B, Ltxt, V, H = args.batch, 100, 29, 512
    amodel = v.TextToAlignTextModel(V, H)
    amodel.load_state_dict({k: torch.from_numpy(np.asarray(t)) for k, t in synth.align_state_dict(V, H, seed=1234).items()})
    vmodel = v.AlignTextToAudioModel(V, H)
    vmodel.load_state_dict({k: torch.from_numpy(np.asarray(t)) for k, t in synth.audio_state_dict(V, H, seed=1234).items()})
    amodel, vmodel = amodel.to(dev).eval(), vmodel.to(dev).eval()
    text = torch.from_numpy(synth.text_tokens(B, Ltxt, V, seed=1234))
    align = torch.from_numpy(synth.synthetic_alignment(B, Ltxt, seed=1234))
    text_d = text.to(dev)
    aligntext, at_len = v.align_batch(text, align)
    at_d = aligntext.to(dev)
    out_frames = float((2 * at_len.double() - 1).sum())          # valid output frames, 10 ms each
    W, K = max(3, args.warmup), max(1, args.steps)
    for _ in range(W):
        amodel(text_d); vmodel.predict(at_d)
    torch.cuda.synchronize()
    n0 = _lib.stats["launches"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        pred = amodel(text_d)
        f0, logspc, codeap = vmodel.predict(at_d)
    e1.record()
    torch.cuda.synchronize()
    ms_eager = e0.elapsed_time(e1) / K
    launches = (_lib.stats["launches"] - n0) // K
    # The same two calls captured once into a CUDA graph (fixed shapes, device-resident inputs): an eager forward pays
    # one host round trip for the embedding's index check plus ~40 Python launches, which a slower host turns into
    # idle gaps between 20-200 us kernels (same kernels: 4.9 ms on one box, 5.7 ms on another).
    outs = {}

    def both():
        outs["align_pred"] = amodel(text_d)
        outs["f0"], outs["logspc"], outs["codeap"] = vmodel.predict(at_d)
    ms, launch = _graph_leg(torch, dev, both, W, K, ms_eager)
    if args.dump_outputs:
        graphed = launch == "CUDA graph replay"
        dump_outputs(args.dump_outputs, outs if graphed else dict(align_pred=pred, f0=f0, logspc=logspc, codeap=codeap))
    # end to end: host text in, host WORLD parameters out, host alignment loop in between
    Ke = max(2, min(K, 5))
    pin = lambda t: torch.empty(t.shape, dtype=t.dtype).pin_memory()
    f0_h, logspc_h, codeap_h, pred_h = pin(f0), pin(logspc), pin(codeap), pin(pred)
    text_p = text.pin_memory()
    t0 = time.perf_counter()
    for _ in range(Ke):
        pred_h.copy_(amodel(text_p.to(dev, non_blocking=True)), non_blocking=True)
        at_h, _ = v.align_batch(text, align)                       # (the benchmark alignment, not exp(pred)-1)
        f0, logspc, codeap = vmodel.predict(at_h.pin_memory().to(dev, non_blocking=True))
        f0_h.copy_(f0, non_blocking=True); logspc_h.copy_(logspc, non_blocking=True); codeap_h.copy_(codeap, non_blocking=True)
        torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / Ke
    print(json.dumps({
        "metric": "tts_output_audio_seconds_per_second", "value": round(out_frames * 0.01 / (ms * 1e-3), 1),
        "unit": "audio-s/s", "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": round(ms, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"tts_en_base: TextToAlignTextModel + AlignTextToAudioModel(29,512), {B} x 100 tokens, "
                               f"aligned text [{B},{aligntext.shape[1]}] -> WORLD [{B},{2 * aligntext.shape[1] - 1},259]",
                   "launch": launch, "eager_ms_per_step": round(ms_eager, 4)},
        "e2e": {"value": round(out_frames * 0.01 / dt, 1), "unit": "audio-s/s", "note": "includes host align_batch, H2D of text and D2H of fp32 WORLD parameters",
                "d2h_bytes_per_step": int(f0_h.numel() + logspc_h.numel() + codeap_h.numel()) * 4},
        "gpu_launches": launches * K, "gpu_launches_per_step": launches}))


def run_tts_v2(args):
    """Secondary workload: the reference's shipped TTS configs (config/align_en_base.yaml + config/tts_en_base.yaml):
    text [B,100] -> TextToAlignText(2 x biLSTM-256) -> host align_batch_v2 (seeded synthetic alignment) ->
    AlignTextToAudio(2 x biLSTM-512, conv / transposed-conv blocks).predict -> WORLD parameters."""
    import numpy as np
    import torch
    import voice100_b200 as v
    from voice100_b200 import _lib, synth
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    B, Ltxt, V = args.batch, 100, 29
    load = lambda m, sd: (m.load_state_dict({k: torch.from_numpy(np.asarray(t)) for k, t in sd.items()}), m.to(dev).eval())[1]
    amodel = load(v.TextToAlignText(V, 2, 256, 2), synth.align_v2_state_dict(V, 2, 256, 2, seed=1234))
    dec = [list(r) for r in synth.TTS_V2_BASE_DECODER]
    vmodel = load(v.AlignTextToAudio(V, 257, 1, 2, 512, dec), synth.audio_v2_state_dict(V, seed=1234))
    text = torch.from_numpy(synth.text_tokens(B, Ltxt, V, seed=1234))
    text_len = torch.full((B,), Ltxt, dtype=torch.int64)
    align = torch.from_numpy(synth.synthetic_alignment(B, Ltxt, seed=1234))
    aligntext, at_len = v.align_batch_v2(text, align, text_len)
    text_d, at_d = text.to(dev), aligntext.to(dev)
    out_frames = float((2 * at_len.double() - 1).sum())
    W, K = max(3, args.warmup), max(1, args.steps)
    for _ in range(W):
        amodel(text_d, text_len); vmodel.predict(at_d, at_len)
    torch.cuda.synchronize()
    n0 = _lib.stats["launches"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        pred, pred_len = amodel(text_d, text_len)
        f0, logspc, codeap = vmodel.predict(at_d, at_len)
    e1.record()
    torch.cuda.synchronize()
    ms_eager = e0.elapsed_time(e1) / K
    launches = (_lib.stats["launches"] - n0) // K

    outs = {}

    def both():
        outs["align_pred"], outs["align_pred_len"] = amodel(text_d, text_len)
        outs["f0"], outs["logspc"], outs["codeap"] = vmodel.predict(at_d, at_len)
    ms, launch = _graph_leg(torch, dev, both, W, K, ms_eager)
    if args.dump_outputs:
        graphed = launch == "CUDA graph replay"
        dump_outputs(args.dump_outputs, outs if graphed else dict(
            align_pred=pred, align_pred_len=pred_len, f0=f0, logspc=logspc, codeap=codeap))
    Ke = max(2, min(K, 5))
    pin = lambda t: torch.empty(t.shape, dtype=t.dtype).pin_memory()
    pred_h, out_h, text_p = pin(pred), (pin(f0), pin(logspc), pin(codeap)), text.pin_memory()
    t0 = time.perf_counter()
    for _ in range(Ke):
        pred, _ = amodel(text_p.to(dev, non_blocking=True), text_len)
        pred_h.copy_(pred, non_blocking=True)
        at_h, at_len_h = v.align_batch_v2(text, align, text_len)      # (the benchmark alignment, not exp(pred)-1)
        outs = vmodel.predict(at_h.pin_memory().to(dev, non_blocking=True), at_len_h)
        for h, d in zip(out_h, outs):
            h.copy_(d, non_blocking=True)
        torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / Ke
    print(json.dumps({
        "metric": "tts_output_audio_seconds_per_second", "value": round(out_frames * 0.01 / (ms * 1e-3), 1),
        "unit": "audio-s/s", "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": round(ms, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"tts v2 (config/align_en_base.yaml + config/tts_en_base.yaml): TextToAlignText + "
                               f"AlignTextToAudio, {B} x 100 tokens, aligned text [{B},{aligntext.shape[1]}] -> "
                               f"WORLD [{B},{2 * int(at_len.max()) - 1},259]",
                   "launch": launch, "eager_ms_per_step": round(ms_eager, 4)},
        "e2e": {"value": round(out_frames * 0.01 / dt, 1), "unit": "audio-s/s",
                "note": "includes the host alignment, H2D of text and D2H of fp32 WORLD parameters",
                "d2h_bytes_per_step": int(sum(t.numel() for t in out_h) * 4 + pred_h.numel() * 4)},
        "gpu_launches": launches * K, "gpu_launches_per_step": launches}))


def run_asr_v2(args):
    """Secondary workload: the architecture of the reference's shipped asr_en_base.yaml (AudioToAlignText: two
    LayerNorm/GELU conv blocks -> 2-layer biLSTM(512) -> Linear) on the headline input shape, B x 15 s clips.
    Same metric as the headline (audio-seconds per second); not the number BASELINE.json quotes."""
    import numpy as np
    import torch
    import voice100_b200 as v
    from voice100_b200 import _lib, synth
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    B, L = args.batch, SAMPLE_RATE * CLIP_SECONDS
    dtype = torch.float16 if args.dtype == "f16" else torch.bfloat16
    settings = [list(r) for r in synth.ASR_V2_BASE_ENCODER]
    model = v.AudioToAlignText(64, settings, 2, 512, args.vocab)
    model.load_state_dict({k: torch.from_numpy(np.asarray(t)) for k, t in
                           synth.asr_v2_state_dict(64, synth.ASR_V2_BASE_ENCODER, 2, 512, args.vocab, seed=1234).items()})
    model = model.to(dev).eval().set_storage_dtype(dtype)
    tr = v.MelSpectrogramAudioTransform().to(dev)
    pipe = v.AsrV2Pipeline(tr, model)
    g = torch.Generator(device=dev).manual_seed(1234)
    wavs = [0.1 * torch.randn((B, L), device=dev, generator=g) for _ in range(2)]   # 2 x 15 MB > nothing; see config
    if args.ragged:
        lengths = torch.from_numpy(synth.ragged_lengths(B, 2 * SAMPLE_RATE, L, seed=1234)).to(dev)
    else:
        lengths = torch.full((B,), L, dtype=torch.int32, device=dev)
    audio_seconds = float(lengths.double().sum()) / SAMPLE_RATE
    W, K = max(3, args.warmup), max(1, args.steps)
    for i in range(W):
        pipe(wavs[i & 1], lengths)
    torch.cuda.synchronize()
    n0 = _lib.stats["launches"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        tokens, out_len = pipe(wavs[i & 1], lengths)
    e1.record()
    torch.cuda.synchronize()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"tokens": tokens, "out_len": out_len})
    ms = e0.elapsed_time(e1) / K
    launches = (_lib.stats["launches"] - n0) // K

    class Tracer:
        def __init__(self):
            self.ev = []

        def before(self, name):
            self._s = torch.cuda.Event(enable_timing=True)
            self._s.record()

        def after(self, name):
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self.ev.append((name, self._s, e))

    _lib.tracer = Tracer()
    pipe(wavs[0], lengths)
    torch.cuda.synchronize()
    ev, _lib.tracer = _lib.tracer.ev, None
    launch_ms = [[name.replace("v100_", ""), round(s.elapsed_time(e), 4)] for name, s, e in ev]
    # end to end: pinned host waveforms in, host tokens out; batch i+1 uploads while batch i computes
    host_wav = [w.cpu().pin_memory() for w in wavs]
    len_h = lengths.cpu().pin_memory()
    for i in range(4):
        pipe.transcribe_host(host_wav[i & 1], len_h, device=dev, chunks=1)
    Ke = max(3, K)
    t0 = time.perf_counter()
    prev = None
    for i in range(Ke):
        ticket = pipe.submit_host(host_wav[i & 1], len_h, device=dev, chunks=1)
        if prev is not None:
            tok_h, _ = prev.result()
        prev = ticket
    tok_h, _ = prev.result()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / Ke
    wav_h = host_wav[0]
    print(json.dumps({
        "metric": "asr_audio_seconds_per_second", "value": round(audio_seconds / (ms * 1e-3), 1), "unit": "audio-s/s",
        "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": round(ms, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": f"asr_en_base v2 (config/asr_en_base.yaml): log-mel + AudioToAlignText(conv k5 x2, "
                               f"biLSTM 2x512, V={args.vocab}) + argmax, {B} x {CLIP_SECONDS} s clips"
                               + (", ragged U[2 s,15 s]" if args.ragged else ""),
                   "l2": "two input batches alternate; every step streams > 1 GB of activations (> L2)"},
        "e2e": {"value": round(audio_seconds / dt, 1), "unit": "audio-s/s",
                "h2d_bytes_per_step": int(wav_h.numel() * 4 + len_h.numel() * 4),
                "d2h_bytes_per_step": int(tok_h.numel() * 8)},
        "gpu_launches": launches * K, "gpu_launches_per_step": launches, "launch_ms": launch_ms}))


class _Tracer:
    """CUDA events around every libv100 entry point (per-kernel device times, one launch at a time)."""

    def __init__(self, torch):
        self.ev, self._torch = [], torch

    def before(self, name):
        self._s = self._torch.cuda.Event(enable_timing=True)
        self._s.record()

    def after(self, name):
        e = self._torch.cuda.Event(enable_timing=True)
        e.record()
        self.ev.append((name, self._s, e))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU,
                    help="utterances per GPU (weak scaling; default: the metric's 256) or in the whole job (--scaling strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch clips per GPU; strong: BASELINE.json configs[1] read literally, ONE batch of "
                         "--batch clips sharded over the ranks with voice100_b200.dist.shard_utterances")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true")
    ap.add_argument("--sustain-seconds", type=float, default=3.0,
                    help="length of the sustained leg (graph replays back to back under the power cap); 0 disables it")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "f16"],
                    help="16-bit storage type of activations/weights (bf16 = the metric's; f16 = same speed, tighter parity)")
    ap.add_argument("--ragged", action="store_true",
                    help="BASELINE.json configs[4]: clip lengths U[2 s, 15 s] padded to the batch maximum (audio-seconds "
                         "then count valid samples only); the default is the metric's fixed 15 s clips")
    ap.add_argument("--vocab", type=int, default=MODEL["vocab_size"], help="44 = asr_ja_phone_base")
    ap.add_argument("--workload", default="asr", choices=["asr", "tts", "asr_v2", "tts_v2"], help="asr = the headline metric")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the arrays the timed path returned in its last step to DIR/<name>.npy "
                         "(inputs are seeded: the same arguments give the same inputs on every run)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "tts":
        return run_tts(args)
    if args.workload == "asr_v2":
        return run_asr_v2(args)
    if args.workload == "tts_v2":
        return run_tts_v2(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    import voice100_b200 as v
    from voice100_b200 import _lib, synth
    from voice100_b200.dist import bind_to_gpu_numa, max_over_ranks, shard_utterances, sum_over_ranks

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the Voice100 hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        bind_to_gpu_numa(local)          # pinned host buffers of each rank live next to its GPU
        dist.init_process_group("nccl", device_id=dev)
    W = max(3, args.warmup)
    K = max(1, args.steps)
    L = SAMPLE_RATE * CLIP_SECONDS
    T_in = 1 + L // 160

    # ---- this rank's utterances ----
    if args.scaling == "strong":
        # one global batch; every rank derives the same length list and the same partition, no communication
        n_global = args.batch
        glob_len = (synth.ragged_lengths(n_global, 2 * SAMPLE_RATE, L, seed=1234) if args.ragged
                    else np.full((n_global,), L, np.int32))
        mine = shard_utterances(glob_len.tolist(), world)[rank]
        lengths_np = glob_len[mine].astype(np.int32)
    else:
        lengths_np = (synth.ragged_lengths(args.batch, 2 * SAMPLE_RATE, L, seed=1234 + rank) if args.ragged
                      else np.full((args.batch,), L, np.int32))
    B = int(len(lengths_np))
    if B == 0:
        raise SystemExit("bench.py: a rank received no utterances (batch smaller than the number of GPUs)")

    cfg = dict(MODEL, vocab_size=args.vocab)
    model = v.AudioToTextCTC(**cfg)
    model.load_state_dict({k: torch.from_numpy(np.asarray(t)) for k, t in synth.asr_state_dict(**cfg, seed=1234).items()})
    model = model.to(dev).eval().set_storage_dtype(torch.float16 if args.dtype == "f16" else torch.bfloat16)
    pipe = v.AsrPipeline(v.MelSpectrogramAudioTransform().to(dev), model)

    # device-resident inputs: int16 PCM of 0.1*N(0,1) and the same samples as fp32 (= pcm / 32768, what torchaudio.load
    # returns); one fp32 batch is 245 MB (> the 126 MB L2) and every step streams ~23 GB of activations through HBM in
    # between, so nothing of the input survives in L2 across steps
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    pcms = [(3276.8 * torch.randn((B, L), device=dev, generator=g)).clamp_(-32768, 32767).to(torch.int16) for _ in range(2)]
    wavs = [p.float() / 32768.0 for p in pcms]
    lengths = torch.from_numpy(lengths_np).to(dev)
    valid_audio_seconds = float(lengths_np.astype(np.float64).sum()) / SAMPLE_RATE      # this rank, per step
    run = pipe.graphed(B, L, device=dev)       # the public API's CUDA-graph form of the whole path (fp32 samples)
    run.waveform.copy_(wavs[0])
    run.lengths.copy_(lengths)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(W):
        run.graph.replay()
    n0 = _lib.stats["launches"]
    pipe(wavs[0], lengths)
    launches_per_step = _lib.stats["launches"] - n0

    sampler = ClockSampler(local)
    # Clock ramp (untimed, on top of the W warm-up steps): a part that sat idle during the host-side setup needs tens of
    # milliseconds of load to reach its boost clock -- one run measured a median of 1740 of 1965 MHz over the timed
    # region with no throttle reason.  Keep replaying until NVML reports >= 97 % of the maximum SM clock under load,
    # stop as soon as the power cap is what holds the clock down, 40 steps at most; the count is reported in `config`.
    ramp_steps = 0
    if sampler.nv is not None and sampler.sm_max:
        while ramp_steps < 40:
            run.graph.replay()
            ramp_steps += 1
            try:
                clk = float(sampler.nv.nvmlDeviceGetClockInfo(sampler.h, sampler.nv.NVML_CLOCK_SM))
                capped = bool(sampler.nv.nvmlDeviceGetCurrentClocksEventReasons(sampler.h) & ClockSampler.BITS["sw_power_cap"])
            except Exception:
                break
            torch.cuda.synchronize()
            if clk >= 0.97 * sampler.sm_max or capped:
                break
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        run.graph.replay()                      # launches_per_step kernels of libv100 per replay, nothing else
    e1.record()
    barrier()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}"),
                     {"tokens": run.tokens, "out_len": run.out_len})
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    ms_max = max_over_ranks(ms, dev)
    audio_seconds_per_step = sum_over_ranks(valid_audio_seconds, dev)
    value = audio_seconds_per_step * K / (ms_max / 1e3)

    # ---- per-kernel device times (separate pass, CUDA events around every launch: kernels run one at a time, at
    #      burst clocks, so their roofline denominators are the BURST peaks) ----
    from voice100_b200 import blocks as _blocks
    work = asr_work_model(B, T_in, MODEL["hidden_size"], MODEL["embed_size"], args.vocab, fused=_blocks.FUSE_EXPAND_DW)
    _lib.tracer = _Tracer(torch)
    prof_steps = min(K, 5)
    for i in range(prof_steps):
        pipe(wavs[i & 1], lengths)
    torch.cuda.synchronize()
    ev, _lib.tracer = _lib.tracer.ev, None
    per_launch = [0.0] * len(work)
    assert len(ev) == prof_steps * len(work), (len(ev), len(work))
    for i, (_, s, e) in enumerate(ev):
        per_launch[i % len(work)] += s.elapsed_time(e) / prof_steps
    peaks = load_peaks()
    classes = {}
    for wk, msl in zip(work, per_launch):
        c = classes.setdefault(wk["kind"], dict(ms=0.0, flops=0.0, bytes=0.0, launches=0))
        c["ms"] += msl; c["flops"] += wk["flops"]; c["bytes"] += wk["bytes"]; c["launches"] += 1
    total_kernel_ms = sum(c["ms"] for c in classes.values())
    roofline_all = {}
    for kind, c in classes.items():
        tf = c["flops"] / (c["ms"] * 1e-3) / 1e12 if c["ms"] > 0 else 0.0
        gbs = c["bytes"] / (c["ms"] * 1e-3) / 1e9 if c["ms"] > 0 else 0.0
        entry = dict(ms_per_step=round(c["ms"], 4), launches=c["launches"], share=round(c["ms"] / total_kernel_ms, 4),
                     tflops=round(tf, 1), gbs=round(gbs, 1))
        if kind in ("gemm", "expand_dw"):
            entry.update(bound="tensor", frac=round(tf / peaks["tf_burst"], 4), frac_burst=round(tf / peaks["tf_burst"], 4),
                         frac_sustained=round(tf / peaks["tf_sustained"], 4), hbm_frac=round(gbs / peaks["hbm_gbs"], 4))
        else:
            entry.update(bound="hbm", frac=round(gbs / peaks["hbm_gbs"], 4))
        roofline_all[kind] = entry
    traffic = {}
    for name in sorted(os.listdir(os.path.join(ROOT, "profiles")), reverse=True):   # newest round first
        if name.endswith("_traffic.json"):
            with open(os.path.join(ROOT, "profiles", name)) as f:
                traffic = json.load(f)
            break
    tcls = traffic.get("per_kernel_class", {})
    for kind, entry in roofline_all.items():
        if kind in tcls:
            entry["dram_bytes_per_step_ncu"] = tcls[kind]["dram_bytes_per_step"]
            entry["algorithmic_bytes_per_step"] = classes[kind]["bytes"]
    dom = max(classes, key=lambda k: classes[k]["ms"])
    dc = classes[dom]
    if dom in ("gemm", "expand_dw"):
        ach = dc["flops"] / dc["launches"] / (dc["ms"] / dc["launches"] * 1e-3) / 1e12
        roofline = dict(kernel="conv_gemm_kernel (tcgen05)" if dom == "gemm" else "expand_dw_kernel (tcgen05 GEMM + mma.sync depthwise epilogue)",
                        bound="tensor", achieved=round(ach, 2),
                        peak=peaks["tf_burst"], unit="TFLOP/s", frac=round(ach / peaks["tf_burst"], 4),
                        frac_burst=round(ach / peaks["tf_burst"], 4), frac_sustained=round(ach / peaks["tf_sustained"], 4),
                        peak_sustained=peaks["tf_sustained"],
                        traffic=(tcls[dom]["dram_bytes_per_launch"] if dom in tcls else None),
                        traffic_note="ncu dram__bytes_read+write per launch, mean over the step's launches of this kernel (%s); "
                                     "algorithmic bytes per launch: %.0f" % (traffic.get("source", "n/a"), dc["bytes"] / dc["launches"]),
                        peak_source=peaks["source"] + "; `frac` divides by the BURST bf16 peak because the launches are "
                                    "event-timed one at a time at burst clocks; frac_sustained is against the power-capped peak",
                        note="mean over the %d launches of this kernel in a step (algorithmic FLOPs / CUDA-event time)" % dc["launches"])
    else:
        ach = dc["bytes"] / (dc["ms"] * 1e-3) / 1e9
        roofline = dict(kernel=dom, bound="hbm", achieved=round(ach, 1), peak=peaks["hbm_gbs"], unit="GB/s",
                        frac=round(ach / peaks["hbm_gbs"], 4),
                        traffic=(tcls[dom]["dram_bytes_per_launch"] if dom in tcls else None), peak_source=peaks["source"])
    step_model = dict(kernel_sum_ms=round(total_kernel_ms, 4), graph_step_ms=round(ms / K, 4),
                      gap_ms=round(ms / K - total_kernel_ms, 4),
                      tflops=round(sum(w["flops"] for w in work) / (ms / K * 1e-3) / 1e12, 1),
                      hbm_gbs=round(sum(w["bytes"] for w in work) / (ms / K * 1e-3) / 1e9, 1))

    # ---- end to end through the public API: pinned HOST waveforms in, HOST tokens out, every batch's H2D/D2H inside
    #      the timed region.  Default input = int16 PCM (what a 16-bit WAV holds; the kernel scales by 1/32768, features
    #      bit-identical to fp32 samples); the fp32 form (twice the H2D bytes) is measured beside it. ----
    host_len = lengths.cpu().pin_memory()
    Ke = max(3, K)

    def e2e_leg(dev_batches, dtype):
        host_wav = [torch.empty((B, L), dtype=dtype).pin_memory() for _ in range(2)]
        for hw, dw in zip(host_wav, dev_batches):
            hw.copy_(dw)
        for i in range(4):
            pipe.transcribe_host(host_wav[i & 1], host_len, device=dev, chunks=1)
        barrier()
        t0 = time.perf_counter()
        prev = None
        for i in range(Ke):
            # streaming use of the public API: batch i uploads/computes while batch i-1's tokens are collected
            ticket = pipe.submit_host(host_wav[i & 1], host_len, device=dev, chunks=1)
            if prev is not None:
                tok_h, len_h = prev.result()
            prev = ticket
        tok_h, len_h = prev.result()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        val = audio_seconds_per_step * Ke / max_over_ranks(dt, dev)
        h2d = B * L * host_wav[0].element_size() + B * 4
        d2h = int(tok_h.numel() * 8 + len_h.numel() * len_h.element_size())
        del host_wav
        return {"value": round(val, 1), "unit": "audio-s/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": Ke, "input": "int16 PCM" if dtype == torch.int16 else "fp32 samples"}

    e2e = e2e_leg(pcms, torch.int16)
    e2e_f32 = e2e_leg(wavs, torch.float32)

    # ---- sustained leg LAST (it heats the part into the power cap; the per-kernel pass above must see burst clocks):
    #      the same graph back to back for >= --sustain-seconds ----
    sustained = None
    if args.sustain_seconds > 0:
        n_sus = max(K, int(args.sustain_seconds / max(ms / K * 1e-3, 1e-6)) + 1)
        s2 = ClockSampler(local)
        s2.start()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for i in range(n_sus):
            run.graph.replay()
        f1.record()
        barrier()
        ms_sus = max_over_ranks(f0.elapsed_time(f1), dev)
        sustained = {"value": round(audio_seconds_per_step * n_sus / (ms_sus / 1e3), 1), "unit": "audio-s/s",
                     "steps": n_sus, "seconds": round(ms_sus / 1e3, 3), "ms_per_step": round(ms_sus / n_sus, 4),
                     "clocks": s2.stop()}

    cpu, eager = None, None
    if rank == 0 and world == 1:
        if not args.no_gpu_eager:
            del pcms, wavs
            torch.cuda.empty_cache()
            eager = gpu_eager_baseline(dev, min(B, 256))
            for k in ("f32", "bf16"):
                if "value" in eager.get(k, {}):
                    eager[k]["this_over_eager"] = round(value / eager[k]["value"], 2)
        if not args.no_cpu_baseline:
            val, cores, sample = cpu_oracle_throughput()
            cpu = {"value": round(val, 2), "unit": "audio-s/s", "cores": cores, "kind": "port", "sample": sample}

    if rank == 0:
        clip_desc = "lengths U[2 s, 15 s] padded with BLANK_AUDIO" if args.ragged else "15 s"
        if args.scaling == "strong":
            wl = (f"AudioToTextCTC(64,512,{args.vocab},512), ONE batch of {args.batch} clips ({clip_desc}) sharded over "
                  f"{world} GPU(s) by shard_utterances")
        elif not args.ragged and args.vocab == MODEL["vocab_size"] and args.batch == BATCH_PER_GPU:
            wl = WORKLOAD
        else:
            wl = f"AudioToTextCTC(64,512,{args.vocab},512), {args.batch} clips per GPU, {clip_desc}"
        print(json.dumps({
            "metric": "asr_audio_seconds_per_second", "value": round(value, 1), "unit": "audio-s/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": round(ms_max / K, 4),
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": wl,
                       "global_batch": args.batch if args.scaling == "strong" else world * B, "clip_seconds": CLIP_SECONDS,
                       "parallelism": f"dp{world} (utterance-sharded, no data-path collective)",
                       "launch": "CUDA graph replay (AsrPipeline.graphed)",
                       "clock_ramp_steps": ramp_steps,
                       "l2": "the 245 MB input batch and every activation tensor exceed the 126 MB L2; ~23 GB stream through HBM per step"},
            "e2e": e2e,
            "e2e_f32": e2e_f32,
            "sustained": sustained,
            "gpu_launches": launches_per_step * K,
            "gpu_launches_per_step": launches_per_step,
            "clocks": clocks,
            "roofline": roofline,
            "roofline_all": roofline_all,
            "step_model": step_model,
            "launch_ms": [[w["kind"], round(m, 4)] for w, m in zip(work, per_launch)],
            "gpu_eager_baseline": eager,
            "cpu_baseline": cpu,
        }))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
