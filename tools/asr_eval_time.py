"""ASR evaluation on the device: v100_ctc_loss and v100_edit_distance alone, against torch's CUDA ctc_loss and a host
DP, and AsrPipeline / AsrV2Pipeline.evaluate against __call__ per step.

    python tools/asr_eval_time.py [--batch 256] [--seconds 15] [--steps 20] [--out profiles/r07_asr_eval.md]

Reports, with the card's name and power limit read in the same run:
  (l) kernels.ctc_loss on raw logits (normalize=True, the log_softmax in the kernel) at batch x (seconds x 50) frames,
      V = 29 and 71, targets of 15 characters a second; torch.nn.functional.ctc_loss on CUDA fp32 log-probabilities of
      the same tensors, alone and with its log_softmax.  CUDA events over `steps` calls after a warm-up.
  (e) kernels.edit_distance on batch pairs of 15 characters a second (hypothesis and reference differ in about 20 % of
      the positions), CUDA events; the same pairs through a pure-Python DP on the host (a few pairs, scaled to the batch).
  (p) evaluate() against __call__() per step, eager, for the v1 model of bench.py (AudioToTextCTC(64, 512, 29, 512)) and
      a v2 model with the base encoder settings (hidden 512).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import voice100_b200 as v  # noqa: E402
from voice100_b200 import kernels as K, synth  # noqa: E402


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


def _targets(rng, batch, n_chars, V):
    lens = rng.integers(int(0.8 * n_chars), n_chars + 1, batch)
    return rng.integers(1, V, (batch, n_chars)), lens


def loss_rows(batch, seconds, steps):
    dev = torch.device("cuda", 0)
    T, L = seconds * 50 + 1, seconds * 15
    rng = np.random.default_rng(0)
    rows = []
    for V in (29, 71):
        g = torch.Generator(device=dev).manual_seed(V)
        logits = 4.0 * torch.randn((T, batch, V), device=dev, generator=g)
        tg, tl = _targets(rng, batch, L, V)
        tg, tl = torch.from_numpy(tg).to(dev), torch.from_numpy(tl).to(dev)
        il = torch.full((batch,), T, dtype=torch.int64, device=dev)
        ours = _events(lambda: v.ctc_loss(logits, tg, il, tl, reduction="none", normalize=True), steps)
        lp = logits.log_softmax(-1)
        theirs = _events(lambda: F.ctc_loss(lp, tg, il, tl, reduction="none"), steps)
        theirs_ls = _events(lambda: F.ctc_loss(logits.log_softmax(-1), tg, il, tl, reduction="none"), steps)
        a = v.ctc_loss(logits, tg, il, tl, reduction="none", normalize=True)
        b = F.ctc_loss(lp.double(), tg, il, tl, reduction="none")
        rel = float(((a.double() - b).abs() / b.abs().clamp_min(1)).max())
        rows.append(dict(V=V, T=T, L=L, ms=ours * 1e3, torch_ms=theirs * 1e3, torch_ls_ms=theirs_ls * 1e3,
                         max_rel_vs_torch_f64=rel))
    return rows


def edit_rows(batch, seconds, steps, host_pairs):
    from ctc_eval_reference import edit_distance_py
    dev = torch.device("cuda", 0)
    n = seconds * 15
    rng = np.random.default_rng(1)
    ref = rng.integers(1, 29, (batch, n))
    hyp = ref.copy()
    flip = rng.random((batch, n)) < 0.2
    hyp[flip] = rng.integers(1, 29, int(flip.sum()))
    h, r = torch.from_numpy(hyp).to(dev), torch.from_numpy(ref).to(dev)
    hl = torch.full((batch,), n - 3, dtype=torch.int32, device=dev)
    rl = torch.full((batch,), n, dtype=torch.int32, device=dev)
    sec = _events(lambda: v.edit_distance(h, hl, r, rl), steps)
    t0 = time.perf_counter()
    for b in range(host_pairs):
        edit_distance_py(hyp[b, :n - 3].tolist(), ref[b, :n].tolist())
    host = (time.perf_counter() - t0) / host_pairs
    return dict(n=n, ms=sec * 1e3, host_ms_per_pair=host * 1e3, host_s_per_batch=host * batch)


def pipeline_rows(batch, seconds, steps):
    import v100_oracle as orc
    dev = torch.device("cuda", 0)
    L = 16000 * seconds
    tr = v.MelSpectrogramAudioTransform().to(dev)
    m1 = v.AudioToTextCTC(64, 512, 29, 512)
    m1.load_state_dict(orc.to_torch_sd(synth.asr_state_dict(64, 512, 29, 512, seed=1234)))
    settings = [list(r) for r in synth.ASR_V2_BASE_ENCODER]
    m2 = v.AudioToAlignText(64, settings, 2, 512, 29)
    m2.load_state_dict({k: torch.from_numpy(x) for k, x in
                        synth.asr_v2_state_dict(64, synth.ASR_V2_BASE_ENCODER, 2, 512, 29, seed=1234).items()},
                       strict=False)
    g = torch.Generator(device=dev).manual_seed(2)
    wav = 0.1 * torch.randn((batch, L), device=dev, generator=g)
    lens = torch.full((batch,), L, dtype=torch.int32, device=dev)
    rng = np.random.default_rng(2)
    tg, tl = _targets(rng, batch, seconds * 15, 29)
    tg, tl = torch.from_numpy(tg).to(dev), torch.from_numpy(tl).to(dev)
    out = {}
    for name, pipe in (("v1", v.AsrPipeline(tr, m1.to(dev).eval())), ("v2", v.AsrV2Pipeline(tr, m2.to(dev).eval()))):
        call = _events(lambda: pipe(wav, lens), steps)
        ids = _events(lambda: pipe.transcribe_ids(wav, lens), steps)
        ev = _events(lambda: pipe.evaluate(wav, lens, tg, tl), steps)
        out[name] = dict(call_ms=call * 1e3, transcribe_ids_ms=ids * 1e3, evaluate_ms=ev * 1e3)
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--seconds", type=int, default=15)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--host-pairs", type=int, default=8)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_asr_eval.md"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("asr_eval_time.py needs a CUDA device")
    card = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          stdout=subprocess.PIPE, text=True).stdout.strip()
    lr = loss_rows(args.batch, args.seconds, args.steps)
    er = edit_rows(args.batch, args.seconds, args.steps, args.host_pairs)
    pr = pipeline_rows(args.batch, args.seconds, args.steps)
    B, S = args.batch, args.seconds
    lines = ["# r07 — ASR evaluation on the device (`v100_ctc_loss`, `v100_edit_distance`, `tools/asr_eval_time.py`)", "",
             f"Card: {card} (name, power limit; read in the same run).  Batch {B} x {S} s, CUDA events over "
             f"{args.steps} calls after a warm-up.", "",
             "## (l) CTC loss, reduction \"none\"", "",
             "`ours`: raw logits in, log_softmax and the forward algorithm in float64 in one kernel.  `torch`: "
             "F.ctc_loss on CUDA fp32 log-probabilities (its forward kernel; `+ log_softmax` adds that launch).", "",
             "| V | frames | target chars | ours ms | torch ms | torch + log_softmax ms | max rel. diff vs torch f64 |",
             "|---|---|---|---|---|---|---|"]
    for r in lr:
        lines.append(f"| {r['V']} | {r['T']} | {int(0.8 * r['L'])}-{r['L']} | {r['ms']:.3f} | {r['torch_ms']:.3f} | "
                     f"{r['torch_ls_ms']:.3f} | {r['max_rel_vs_torch_f64']:.1e} |")
    lines += ["", "## (e) edit distance", "",
              f"- device, {B} pairs of {er['n'] - 3} x {er['n']} ids: {er['ms']:.3f} ms",
              f"- host, pure-Python DP: {er['host_ms_per_pair']:.2f} ms a pair = {er['host_s_per_batch']:.2f} s a batch "
              f"(one core)", "",
              "## (p) evaluate() against __call__(), eager, per step", "",
              "| model | __call__ ms | transcribe_ids ms | evaluate ms |", "|---|---|---|---|"]
    for name, r in pr.items():
        lines.append(f"| {name} | {r['call_ms']:.3f} | {r['transcribe_ids_ms']:.3f} | {r['evaluate_ms']:.3f} |")
    text = "\n".join(lines) + "\n"
    print(text)
    with open(args.out, "w") as f:
        f.write(text)
    print(json.dumps(dict(card=card, loss=lr, edit=er, pipelines=pr)))


if __name__ == "__main__":
    main()
