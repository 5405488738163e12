"""Text -> WORLD parameters at 256 x 100 tokens: the stepwise path with the host alignment against the device pipelines.

    python tools/tts_pipeline_time.py [--batch 256] [--steps 20] [--json OUT.json]

For v1 (tts_en_base: TextToAlignTextModel + AlignTextToAudioModel, hidden 512) and v2 (align_en_base + tts_en_base:
TextToAlignText + AlignTextToAudio) it reports, per batch:
  (a) stepwise: align model -> torch.exp - 1 -> D2H -> align_batch[_v2] -> H2D -> predict, wall clock ending in a
      synchronise (what a user had to write before TtsPipeline / TtsV2Pipeline);
  (b) the pipeline, eager (one plan round trip for the lengths);
  (c) the pipeline captured as one CUDA graph with max_frames = the batch's longest aligned text, CUDA events;
  (m) the two models alone, captured as one CUDA graph on a fixed aligned text (the bench's measurement), CUDA events;
  (k) v100_tts_align alone (log1p input, fill at max_frames), CUDA events over 5 replays of a graph of 200 launches;
and whether (a) and (b) agree bit for bit.  The align heads are scaled down and biased to log1p((0.5, 2.0)), so the
predicted durations are about 2.5 frames a token and 260 frames an utterance, the scale of the bench's synthetic
alignment.  The card's name, power limit and maximum SM clock are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import voice100_b200 as v  # noqa: E402
from voice100_b200 import kernels as K, synth  # noqa: E402

V = 29


def _load(model, sd, dev):
    model.load_state_dict({k: torch.from_numpy(np.asarray(t)) for k, t in sd.items()})
    return model.to(dev).eval()


def _realistic_head(sd, key, scale=0.1):
    sd = dict(sd)
    sd[key + ".weight"] = (np.asarray(sd[key + ".weight"]) * scale).astype(np.float32)
    sd[key + ".bias"] = np.log1p(np.array([0.5, 2.0], np.float32)).astype(np.float32)
    return sd


def _wall(fn, steps):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / steps * 1e3


def _events(fn, steps):
    fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def _graph(fn, dev):
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for _ in range(2):
            fn()
    torch.cuda.current_stream(dev).wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g


def _same(a, b):
    return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


@torch.no_grad()
def run(version, B, L, steps, dev):
    text = torch.from_numpy(synth.text_tokens(B, L, V, seed=2024))
    text_len = torch.full((B,), L, dtype=torch.int32)
    text_d, text_len_d = text.to(dev), text_len.to(dev)
    if version == 1:
        H = 512
        amodel = _load(v.TextToAlignTextModel(V, H), _realistic_head(synth.align_state_dict(V, H, seed=1234),
                                                                     "layers.4"), dev)
        vmodel = _load(v.AlignTextToAudioModel(V, H), synth.audio_state_dict(V, H, seed=1234), dev)
        pipe = v.TtsPipeline(amodel, vmodel)

        def stepwise():
            align = torch.exp(amodel(text_d)) - 1
            at, at_len = v.align_batch(text, align.cpu(), text_len)
            return vmodel.predict(at.to(dev)), at_len

        def models(at_d, at_len):
            amodel(text_d)
            return vmodel.predict(at_d)
        pred_head = lambda: amodel._head_ncw(text_d).data.transpose(1, 2)[:, :L]
    else:
        amodel = _load(v.TextToAlignText(V, 2, 256, 2), _realistic_head(synth.align_v2_state_dict(V, 2, 256, 2,
                                                                                                  seed=1234), "dense"), dev)
        dec = [list(r) for r in synth.TTS_V2_BASE_DECODER]
        vmodel = _load(v.AlignTextToAudio(V, 257, 1, 2, 512, dec), synth.audio_v2_state_dict(V, seed=1234), dev)
        pipe = v.TtsV2Pipeline(amodel, vmodel)

        def stepwise():
            align, _ = amodel.predict(text_d, text_len)
            at, at_len = v.align_batch_v2(text, align.cpu(), text_len)
            return vmodel.predict(at.to(dev), at_len), at_len

        def models(at_d, at_len):
            amodel(text_d, text_len)
            return vmodel.predict(at_d, at_len)

        def pred_head():
            y, tm = amodel._head_tm(text_d, text_len_d)
            return torch.as_strided(y.data, (tm.B, tm.T, 2), (1, tm.Bp, y.pitch))
    rule = version

    (f0a, spa, apa), at_len = stepwise()
    max_frames = int(at_len.max())
    f0b, spb, apb, frame_len, status = pipe(text_d, text_len_d)
    torch.cuda.synchronize()
    exact = _same(f0a, f0b) and _same(spa, spb) and _same(apa, apb) and torch.equal(frame_len.cpu(), 2 * at_len - 1)

    ms_a = _wall(stepwise, steps)
    ms_b = _wall(lambda: pipe(text_d, text_len_d), steps)
    graphed = pipe.graphed(B, L, max_frames, device=dev)
    ms_c = _events(lambda: graphed.graph.replay(), steps)
    graphed(text_d, text_len_d)
    torch.cuda.synchronize()
    c_equal = all(_same(x, y) for x, y in zip(graphed.outputs[:3], (f0b, spb, apb)))

    fixed = torch.from_numpy(synth.synthetic_alignment(B, L, seed=1234))       # the bench's synthetic alignment
    at_d, at_len_fixed = (v.align_batch if version == 1 else v.align_batch_v2)(text, fixed, text_len)
    at_d = at_d.to(dev)
    g_models = _graph(lambda: models(at_d, at_len_fixed), dev)
    ms_m = _events(lambda: g_models.replay(), steps)

    # 200 launches captured back to back, so that the host cost of a Python call does not hide the kernel's
    head = pred_head()
    g_k = _graph(lambda: [K.tts_align(text_d, head, text_len_d, rule, 5, 5, max_frames, True) for _ in range(200)], dev)
    ms_k = _events(lambda: g_k.replay(), 5) / 200
    return {
        "version": version, "batch": B, "tokens": L, "max_frames": max_frames,
        "mean_frames": round(float(at_len.float().mean()), 1),
        "frames_per_token": round(float((at_len.float() - 10).mean()) / L, 3),
        "ms_a_stepwise_host_align": round(ms_a, 3), "ms_b_pipeline_eager": round(ms_b, 3),
        "ms_c_pipeline_graphed": round(ms_c, 3), "ms_models_graphed_fixed_alignment": round(ms_m, 3),
        "models_fixed_alignment_frames": int(at_d.shape[1]),
        "ms_tts_align_kernel": round(ms_k, 4), "a_equals_b_bitwise": bool(exact), "c_equals_b_bitwise": bool(c_equal),
        "status_nonzero": int((status != 0).sum()),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--tokens", type=int, default=100)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tts_pipeline_time.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                          capture_output=True, text=True).stdout.strip()
    res = {"card": card, "results": [run(ver, args.batch, args.tokens, args.steps, dev) for ver in (1, 2)]}
    print(json.dumps(res, indent=1))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
