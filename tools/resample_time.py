"""Resampling on the device: v100_resample alone, torchaudio's resample on the same GPU and on the host, and the cost of
a 44.1 kHz input inside the graphed v1 ASR step.

    python tools/resample_time.py [--batch 256] [--seconds 15] [--steps 20] [--out profiles/r05_resample.md]

Reports, with the card's name and power limit read in the same run:
  (k) kernels.resample alone at batch x seconds of input for 48 / 44.1 / 22.05 kHz -> 16 kHz (fp32 and int16 input) and
      16 -> 48 kHz (fp32): CUDA events over `steps` calls after a warm-up.  Bytes are the input and output rows (the
      ~40 KB table is ignored); FLOPs are 2 x the packed taps of every output sample.  The bound is the larger of
      bytes / 7.7 TB/s and FLOPs / (148 SMs x 128 FMA/clk x 2 x the SM clock nvidia-smi reports right after the timed
      loop); each row repeats with the packed table read through the read-only path instead of shared memory
      (V100_RESAMPLE_TAPS=ldg, a child process).
  (t) torchaudio.functional.resample 44.1 -> 16 kHz on CUDA tensors of the same batch (CUDA events) and on the host
      with all threads (wall clock, a smaller batch), as input audio seconds per second.
  (g) the graphed v1 ASR step (asr_en_base, bench.py's model) on int16 PCM at 44.1 kHz against the same batch at 16 kHz.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import voice100_b200 as v  # noqa: E402
from voice100_b200 import data_modules as dm, kernels as K, synth  # noqa: E402

HBM = 7.7e12
CASES = [(48000, 16000, "f32"), (48000, 16000, "i16"), (44100, 16000, "f32"), (44100, 16000, "i16"),
         (22050, 16000, "f32"), (22050, 16000, "i16"), (16000, 48000, "f32")]


def _events(fn, steps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps * 1e-3


def _sm_clock_mhz():
    r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits"],
                       stdout=subprocess.PIPE, text=True)
    return float(r.stdout.strip().splitlines()[0])


def kernel_rows(batch, seconds, steps):
    dev = torch.device("cuda", 0)
    rows = []
    for a, b, kind in CASES:
        L = a * seconds
        g = torch.Generator(device=dev).manual_seed(a)
        pcm = torch.randint(-8000, 8000, (batch, L), device=dev, dtype=torch.int16, generator=g)
        x = pcm if kind == "i16" else pcm.float() / 32768.0
        lens = torch.full((batch,), L, dtype=torch.int32, device=dev)
        tab = dm.resample_table(a, b, device=dev)
        L_out = dm.resampled_length(L, a, b)
        sec = _events(lambda: K.resample(x, lens, tab, L_out), steps)
        clk = _sm_clock_mhz()
        del x, pcm
        nbytes = batch * (L * (2 if kind == "i16" else 4) + L_out * 4)
        flops = 2.0 * batch * (L_out / tab.n) * tab.taps.numel()
        peak_flops = 148 * 128 * 2 * clk * 1e6
        bound = max(nbytes / HBM, flops / peak_flops)
        rows.append(dict(orig=a, new=b, input=kind, ms=sec * 1e3, gbs=nbytes / sec / 1e9, tflops=flops / sec / 1e12,
                         sm_mhz=clk, bound_by="HBM" if nbytes / HBM >= flops / peak_flops else "FMA",
                         share=bound / sec, in_audio_s_per_s=batch * seconds / sec))
    return rows


def torchaudio_rows(batch, seconds, steps, host_batch):
    import torchaudio.functional as AF
    dev = torch.device("cuda", 0)
    a, b = 44100, 16000
    x = torch.randn((batch, a * seconds), device=dev) * 0.1
    sec = _events(lambda: AF.resample(x, a, b), max(2, steps // 4))
    del x
    xh = torch.randn((host_batch, a * seconds)) * 0.1
    AF.resample(xh[:1], a, b)
    t0 = time.perf_counter()
    AF.resample(xh, a, b)
    host = time.perf_counter() - t0
    return dict(gpu_ms=sec * 1e3, gpu_audio_s_per_s=batch * seconds / sec, host_threads=torch.get_num_threads(),
                host_batch=host_batch, host_s=host, host_audio_s_per_s=host_batch * seconds / host)


def asr_rows(batch, seconds, steps):
    import v100_oracle as orc
    dev = torch.device("cuda", 0)
    model = v.AudioToTextCTC(64, 512, 29, 512)
    model.load_state_dict(orc.to_torch_sd(synth.asr_state_dict(64, 512, 29, 512, seed=1234)))
    pipe = v.AsrPipeline(v.MelSpectrogramAudioTransform().to(dev), model.to(dev).eval())
    out = {}
    for rate in (16000, 44100):
        L = rate * seconds
        g = torch.Generator(device=dev).manual_seed(rate)
        pcm = torch.randint(-3277, 3277, (batch, L), device=dev, dtype=torch.int16, generator=g)
        lens = torch.full((batch,), L, dtype=torch.int32, device=dev)
        run = pipe.graphed(batch, L, dev, torch.int16, sample_rate=rate)
        run(pcm, lens)
        sec = _events(run.graph.replay, steps)
        out[rate] = dict(ms=sec * 1e3, audio_s_per_s=batch * seconds / sec)
        del run, pcm
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--seconds", type=int, default=15)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--host-batch", type=int, default=8)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_resample.md"))
    ap.add_argument("--kernels-json", action="store_true", help="print (k) as JSON and exit (used for the ldg child)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("resample_time.py needs a CUDA device")
    if args.kernels_json:
        print(json.dumps(kernel_rows(args.batch, args.seconds, args.steps)))
        return
    card = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          stdout=subprocess.PIPE, text=True).stdout.strip()
    rows = kernel_rows(args.batch, args.seconds, args.steps)
    child = subprocess.run([sys.executable, os.path.abspath(__file__), "--kernels-json", "--batch", str(args.batch),
                            "--seconds", str(args.seconds), "--steps", str(args.steps)],
                           env=dict(os.environ, V100_RESAMPLE_TAPS="ldg"), stdout=subprocess.PIPE, text=True, check=True)
    ldg = json.loads(child.stdout.strip().splitlines()[-1])
    ta = torchaudio_rows(args.batch, args.seconds, args.steps, args.host_batch)
    asr = asr_rows(args.batch, args.seconds, args.steps)

    B, S = args.batch, args.seconds
    lines = [f"# r05 — resampling on the device (`v100_resample`, `tools/resample_time.py`)", "",
             f"Card: {card} (name, power limit; read in the same run).  Batch {B} x {S} s of input, CUDA events over "
             f"{args.steps} calls after a warm-up; the input is larger than L2 at every rate.", "",
             "## (k) the kernel alone", "",
             "Bytes: input + output rows.  FLOPs: 2 x packed taps per output.  Bound: the larger of bytes / 7.7 TB/s "
             "and FLOPs / (148 x 128 FMA/clk x 2 x SM clock read by nvidia-smi right after the loop).  "
             "`ldg`: the same kernel reading the packed table through the read-only path instead of shared memory.", "",
             "| rate | input | ms | GB/s | TFLOP/s | SM MHz | bound by | share of bound | input audio-s/s | ldg ms |",
             "|---|---|---|---|---|---|---|---|---|---|"]
    for r, l in zip(rows, ldg):
        lines.append(f"| {r['orig']} → {r['new']} | {r['input']} | {r['ms']:.3f} | {r['gbs']:.0f} | {r['tflops']:.2f} | "
                     f"{r['sm_mhz']:.0f} | {r['bound_by']} | {r['share']:.2f} | {r['in_audio_s_per_s']:.3g} | "
                     f"{l['ms']:.3f} |")
    lines += ["", "## (t) torchaudio.functional.resample, 44.1 → 16 kHz, fp32", "",
              f"- same GPU, CUDA tensors, {B} x {S} s: {ta['gpu_ms']:.2f} ms = {ta['gpu_audio_s_per_s']:.3g} input audio-s/s",
              f"- host, {ta['host_threads']} threads, {ta['host_batch']} x {S} s: {ta['host_s']:.2f} s = "
              f"{ta['host_audio_s_per_s']:.3g} input audio-s/s", "",
              "## (g) graphed v1 ASR step (asr_en_base), int16 PCM input", "",
              "| input rate | step ms | audio-s/s |", "|---|---|---|"]
    for rate, r in asr.items():
        lines.append(f"| {rate} | {r['ms']:.3f} | {r['audio_s_per_s']:.3g} |")
    lines += ["", f"The 44.1 kHz step costs {asr[44100]['ms'] - asr[16000]['ms']:.3f} ms more than the 16 kHz one "
              "(the resampling kernel plus its fp32 16 kHz round trip).", ""]
    text = "\n".join(lines)
    print(text)
    with open(args.out, "w") as f:
        f.write(text)
    print(json.dumps(dict(card=card, kernels=rows, ldg=ldg, torchaudio=ta, asr=asr)))


if __name__ == "__main__":
    main()
