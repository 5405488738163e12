"""Time WORLD analysis on the device (v100_world_analyze via WORLDVocoder.encode_batch).

    python tools/world_analysis_time.py [--batch 256] [--seconds 15] [--iters 10] [--out DIR]

- Input: `--batch` utterances of `--seconds` s of the speech-like signal of tests/world_analysis_data.py (8 distinct
  clips, repeated), fp32 at 16 kHz, plus one 22.05 kHz case (the same clips resampled on the device first).
- Timing: CUDA events around the whole call, eager and replayed as a CUDA graph, after warm-up; per-kernel times from
  torch.profiler in a separate pass.
- Bounds: float64 operations and bytes from the shapes and the number of voiced / analysed frames, over the data
  sheet's per-GPU FP64 rate (37 TFLOP/s for HGX B200) and HBM bandwidth (7.7 TB/s).
- Host reference: the numpy restatement (oracle/world_analysis.py, not pyworld) on every host thread.
Prints the card's name and power limit beside the numbers.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

FP64_PEAK = 37e12
HBM_PEAK = 7.7e12


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip().splitlines()[0]
        return q
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def clips(n_distinct, seconds, seed=0):
    from world_analysis_data import speechlike
    return [speechlike(int(seconds * 16000), seed + i) for i in range(n_distinct)]


def bounds(B, L, f0, d4c_frames):
    """float64 operations and HBM bytes of one call from the shapes and frame counts."""
    T = L // 160 + 1
    voiced = int((f0 > 0).sum())
    fft = lambda n: 5.0 * n * math.log2(n)
    flops = {
        "DIO filters": B * (2.0 * 641 * (L + 320) + 2 * 2.0 * 992 * L),
        "StoneMask": voiced * fft(2048),
        "CheapTrick": B * T * 3 * fft(512),
        "D4C": voiced * fft(2048) + d4c_frames * 4 * fft(2048),
    }
    byts = {
        "DIO filters": B * (4.0 * L + 8.0 * (L + 320) * (1 + 2 * 7) + 8.0 * 28 * L / 4),
        "StoneMask": B * T * 12.0,
        "CheapTrick": B * T * (257 * 4 + 766 * 8),
        "D4C": d4c_frames * 5290 * 8.0 + B * T * 4,
    }
    return flops, byts


def host_worker(x):
    import world_analysis as A
    t = time.perf_counter()
    A.encode(x)
    return time.perf_counter() - t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--seconds", type=float, default=15.0)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--host-seconds", type=float, default=3.0)
    ap.add_argument("--out", default=None, help="directory for world_analysis_time.json (default: print only)")
    a = ap.parse_args()
    import torch
    import voice100_b200 as v
    if not torch.cuda.is_available():
        raise SystemExit("world_analysis_time.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"card": card(), "batch": a.batch, "seconds": a.seconds}
    print("card:", res["card"])
    base = clips(8, a.seconds)
    L = len(base[0])
    x = torch.from_numpy(np.stack([base[i % 8] for i in range(a.batch)])).to(dev)
    ln = torch.full((a.batch,), L, dtype=torch.int32, device=dev)
    voc = v.WORLDVocoder()

    def timed(fn, iters):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ts = []
        for _ in range(iters):
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))

    out = voc.encode_batch(x, ln)
    torch.cuda.synchronize()
    audio_s = a.batch * a.seconds
    eager = timed(lambda: voc.encode_batch(x, ln), a.iters)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        voc.encode_batch(x, ln)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        voc.encode_batch(x, ln)
    graph = timed(g.replay, a.iters)
    res["eager_ms"], res["graph_ms"] = eager, graph
    res["audio_s_per_s_eager"] = audio_s / (eager[0] / 1e3)
    res["audio_s_per_s_graph"] = audio_s / (graph[0] / 1e3)
    print(f"16 kHz, {a.batch} x {a.seconds} s: eager {eager[0]:.1f} ms (min {eager[1]:.1f}, max {eager[2]:.1f}), "
          f"graph {graph[0]:.1f} ms -> {res['audio_s_per_s_graph']:.0f} audio-s/s")

    # 22.05 kHz: the same clips resampled to 22.05 kHz on the device, then encode_batch(sample_rate=22050)
    x22, l22 = v.resample(x, 16000, 22050, lengths=ln)
    t22 = timed(lambda: voc.encode_batch(x22, l22, sample_rate=22050), a.iters)
    res["sr22050_ms"] = t22
    print(f"22.05 kHz input (resample + analysis): {t22[0]:.1f} ms -> {audio_s / (t22[0] / 1e3):.0f} audio-s/s")

    # per-kernel times (profiler in a pass of its own)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            voc.encode_batch(x, ln)
        torch.cuda.synchronize()
    per = {}
    for ev in prof.key_averages():
        if "wa_" in ev.key:
            name = "wa_" + ev.key.split("wa_")[1].split("(")[0]
            per[name] = per.get(name, 0.0) + ev.device_time_total / 3 / 1e3
    f0 = out[0].cpu().numpy()
    codeap = out[2].cpu().numpy()
    d4c_frames = int((codeap[..., 0] < -1e-9).sum())
    flops, byts = bounds(a.batch, L, f0, d4c_frames)
    stage = {"DIO filters": ["wa_prep", "wa_lowcut", "wa_bands", "wa_scan", "wa_contour", "wa_fix"],
             "StoneMask": ["wa_stonemask"], "CheapTrick": ["wa_cheaptrick", "wa_draws"],
             "D4C": ["wa_lovetrain", "wa_d4c"]}
    res["kernels_ms"] = per
    res["stages"] = {}
    for k, names in stage.items():
        ms = sum(t for n, t in per.items() if any(n.startswith(m) for m in names))
        lb = max(flops[k] / FP64_PEAK, byts[k] / HBM_PEAK) * 1e3
        which = "FP64" if flops[k] / FP64_PEAK > byts[k] / HBM_PEAK else "HBM"
        res["stages"][k] = dict(ms=ms, gflop=flops[k] / 1e9, gbyte=byts[k] / 1e9, bound_ms=lb, bound=which,
                                share=lb / ms if ms else None)
        print(f"  {k:12s} {ms:8.2f} ms  {flops[k] / 1e9:9.1f} GFLOP  {byts[k] / 1e9:7.2f} GB  "
              f"bound {lb:6.2f} ms ({which})  share of peak {lb / ms if ms else float('nan'):.3f}")
    for n, t in sorted(per.items(), key=lambda kv: -kv[1]):
        print(f"    {n:40s} {t:8.2f} ms")

    # host reference: the numpy restatement on every host thread
    nproc = os.cpu_count() or 1
    hx = [c[:int(a.host_seconds * 16000)] for c in clips(nproc, a.host_seconds, seed=100)]
    t0 = time.perf_counter()
    with ProcessPoolExecutor(nproc) as ex:
        list(ex.map(host_worker, hx))
    dt = time.perf_counter() - t0
    res["host_threads"] = nproc
    res["host_audio_s_per_s"] = nproc * a.host_seconds / dt
    print(f"host reference (numpy restatement, not pyworld), {nproc} threads: {res['host_audio_s_per_s']:.1f} audio-s/s")
    if a.out is None:
        return
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "world_analysis_time.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
