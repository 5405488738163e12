"""WORLD synthesis on the device: vocoder throughput on the v1 256 x 100-token pipeline output, and text -> PCM against
text -> WORLD parameters.

    python tools/world_time.py [--batch 256] [--tokens 100] [--steps 10] [--oracle-utts 64] [--json OUT.json]

Reports, with the card's name, power limit and maximum SM clock read in the same run:
  (v) kernels.world_synthesize alone on the v1 pipeline's WORLD parameters (tts_en_base shapes, align head biased to
      about 2.5 frames a token as in tools/tts_pipeline_time.py): CUDA events over `steps` calls, as output audio
      seconds per second, with the pulse count and the split between v100_world_timebase and the rest;
  (n) v100_world_noise for a 60 s table (960,000 values), CUDA events, one call;
  (g) for v1 and v2 (AlignTextToAudio, 257 bins): the pipeline captured as one CUDA graph, text -> WORLD parameters and
      text -> PCM, at max_frames = the batch's longest aligned text, CUDA events over graph replays;
  (o) the float64 numpy restatement oracle/world.py (NOT pyworld) on `--oracle-utts` utterances of (v), one process per
      host thread, wall clock, as output audio seconds per second.
"""
import argparse
import json
import multiprocessing as mp
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
from voice100_b200 import _lib, kernels as K, synth  # noqa: E402

V = 29


def _load(model, sd, dev):
    model.load_state_dict({k: torch.from_numpy(np.asarray(t)) for k, t in sd.items()})
    return model.to(dev).eval()


def _realistic_head(sd, key, scale=0.1):
    sd = dict(sd)
    sd[key + ".weight"] = (np.asarray(sd[key + ".weight"]) * scale).astype(np.float32)
    sd[key + ".bias"] = np.log1p(np.array([0.5, 2.0], np.float32)).astype(np.float32)
    return sd


def _events(fn, steps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def _pipes(dev):
    H = 512
    a1 = _load(v.TextToAlignTextModel(V, H), _realistic_head(synth.align_state_dict(V, H, seed=1234), "layers.4"), dev)
    m1 = _load(v.AlignTextToAudioModel(V, H), synth.audio_state_dict(V, H, seed=1234), dev)
    a2 = _load(v.TextToAlignText(V, 2, 256, 2), _realistic_head(synth.align_v2_state_dict(V, 2, 256, 2, seed=1234),
                                                                "dense"), dev)
    dec = [list(r) for r in synth.TTS_V2_BASE_DECODER]
    m2 = _load(v.AlignTextToAudio(V, 257, 1, 2, 512, dec), synth.audio_v2_state_dict(V, seed=1234), dev)
    return {1: v.TtsPipeline(a1, m1), 2: v.TtsV2Pipeline(a2, m2)}


def _oracle_one(args):
    import world as W
    f0, sp, ap = args
    t0 = time.perf_counter()
    y = W.synthesize(f0, sp, ap)
    return len(y), time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--tokens", type=int, default=100)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--oracle-utts", type=int, default=64)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("world_time.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                          capture_output=True, text=True).stdout.strip()
    B, L = args.batch, args.tokens
    text = torch.from_numpy(synth.text_tokens(B, L, V, seed=2024)).to(dev)
    text_len = torch.full((B,), L, dtype=torch.int32, device=dev)
    pipes = _pipes(dev)
    res = {"card": card, "batch": B, "tokens": L}

    with torch.no_grad():
        f0, logspc, codeap, frame_len, _ = pipes[1](text, text_len)
        torch.cuda.synchronize()
        K.world_noise(160 * f0.shape[1], dev)
        wav, wav_len, status = K.world_synthesize(f0, logspc, codeap, frame_len)
        tb = K.world_timebase(f0, logspc, codeap, frame_len)
        audio_s = float(wav_len.sum()) / K.WORLD_FS
        ms_total = _events(lambda: K.world_synthesize(f0, logspc, codeap, frame_len), args.steps)
        ms_tb = _events(lambda: K.world_timebase(f0, logspc, codeap, frame_len), args.steps)
        res["vocoder"] = {
            "frames_T": int(f0.shape[1]), "mean_frames": round(float(frame_len.float().mean()), 1),
            "output_audio_s": round(audio_s, 1), "pulses": int(tb["head"][:, 3].sum()),
            "status_nonzero": int((status != 0).sum()),
            "ms_total": round(ms_total, 3), "ms_timebase": round(ms_tb, 3), "ms_synthesis": round(ms_total - ms_tb, 3),
            "output_audio_s_per_s": round(audio_s / (ms_total / 1e3), 0),
        }
        n60 = 60 * K.WORLD_FS
        tab = torch.empty(n60, dtype=torch.float64, device=dev)
        stream = torch.cuda.current_stream().cuda_stream
        res["noise_60s_ms"] = round(_events(lambda: _lib.call("v100_world_noise", tab.data_ptr(), n60, stream), 1), 2)

        res["graphed"] = []
        for ver, pipe in pipes.items():
            _, _, _, fl, _ = pipe(text, text_len)
            max_frames = (int(fl.max()) + 1) // 2
            g_world = pipe.graphed(B, L, max_frames)
            g_pcm = pipe.graphed(B, L, max_frames, waveform=True)
            g_world(text, text_len)
            g_pcm(text, text_len)
            ms_w = _events(lambda: g_world.graph.replay(), args.steps)
            ms_p = _events(lambda: g_pcm.graph.replay(), args.steps)
            wl = g_pcm.outputs[1]
            secs = float(wl.sum()) / K.WORLD_FS
            res["graphed"].append({"version": ver, "max_frames": max_frames, "ms_text_to_world": round(ms_w, 3),
                                   "ms_text_to_pcm": round(ms_p, 3), "output_audio_s": round(secs, 1),
                                   "pcm_audio_s_per_s": round(secs / (ms_p / 1e3), 0)})
            del g_world, g_pcm

    n = min(args.oracle_utts, B)
    jobs = [(f0[b, :int(frame_len[b])].cpu().numpy(), logspc[b, :int(frame_len[b])].cpu().numpy(),
             codeap[b, :int(frame_len[b])].cpu().numpy()) for b in range(n)]
    threads = os.cpu_count() or 1
    with mp.get_context("spawn").Pool(threads) as pool:
        pool.map(_oracle_one, jobs[:threads])                 # warm: imports and each process's noise table
        t0 = time.perf_counter()
        out = pool.map(_oracle_one, jobs)
        wall = time.perf_counter() - t0
    secs = sum(o[0] for o in out) / K.WORLD_FS
    res["numpy_restatement"] = {"label": "oracle/world.py float64 numpy restatement, not pyworld",
                                "host_threads": threads, "utterances": n, "output_audio_s": round(secs, 1),
                                "wall_s": round(wall, 2), "output_audio_s_per_s": round(secs / wall, 1)}
    print(json.dumps(res, indent=1))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
