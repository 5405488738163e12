"""TTS text alignment on the device (v100_tts_align, align_frames) and the text -> WORLD pipelines built on it
(TtsPipeline, TtsV2Pipeline).

The alignment is integer work whose semantics are pinned by host code: TextToAlignTextModel.align / _align_one /
align_batch (rule 1), TextToAlignText.align / align_batch_v2 (rule 2), and the reference's own outputs in
tests/golden/align_edges.json.  Every comparison here is exact: frame ids, lengths, and the pipelines' WORLD
parameters as bit patterns."""
import json
import math
import os

import numpy as np
import pytest
import torch

import voice100_b200 as v
from voice100_b200 import _lib, kernels as K, synth
from voice100_b200.tts import _align_one
from helpers import GOLDEN

pytestmark = pytest.mark.gpu
DEV = "cuda"
V = 29
FAILED_AS = {K.ALIGN_INDEX: IndexError, K.ALIGN_NEGATIVE: RuntimeError, K.ALIGN_NAN: ValueError,
             K.ALIGN_INF: OverflowError}


def _rng(seed):
    return np.random.Generator(np.random.PCG64(seed))


def _host_rule1(text, a, head=5, tail=5):
    """(frames, None) or (None, exception class) from the reference loop for one utterance."""
    try:
        total = head + int(torch.sum(torch.from_numpy(np.ascontiguousarray(a)))) + tail
        return _align_one(list(map(int, text)), a.astype(np.float64).tolist(), total, head), None
    except (IndexError, RuntimeError, ValueError, OverflowError) as exc:
        return None, type(exc)


def _host_rule2(text, a, head=5, tail=5):
    if len(text) == 0:
        return [0] * (head + tail), None
    try:
        return v.TextToAlignText.align(torch.tensor(np.asarray(text), dtype=torch.int64), torch.from_numpy(a),
                                       head, tail).tolist(), None
    except (IndexError, RuntimeError, ValueError, OverflowError) as exc:
        return None, type(exc)


def _sum_straddles_integer(a, rule):
    """True when the exact float64 sum and the CPU torch.sum of this utterance's entries truncate to different
    integers: the one case in which the device's total (fp32 rounding of the sequential fp64 sum) may differ."""
    t = torch.from_numpy(np.ascontiguousarray(a))
    exact = math.fsum(a.astype(np.float64).ravel().tolist())
    cpu = torch.sum(t)
    if rule == 2:
        exact -= float(a[0, 0])
        cpu = cpu - t[0, 0]
    return math.trunc(exact) != int(cpu) or math.trunc(float(np.float32(exact))) != int(cpu)


def _check_against_host(text, align, text_len, rule, max_frames):
    """Capacity-mode call (no raise) on the whole batch, then every utterance against the host loop."""
    host = _host_rule1 if rule == 1 else _host_rule2
    at, n, status = v.align_frames(text.to(DEV), align.to(DEV), text_len.to(DEV), rule=rule, max_frames=max_frames)
    at, n, status = at.cpu(), n.cpu(), status.cpu()
    n_ok = n_skipped = 0
    for b in range(text.shape[0]):
        L = int(text_len[b])
        a = align[b, :L].numpy()
        ref, exc = host(text[b, :L].tolist(), a)
        st = int(status[b])
        if exc is not None:
            assert st in FAILED_AS and FAILED_AS[st] is exc, (b, st, exc)
            assert int(n[b]) == 0 and (at[b] == 0).all()
            continue
        if st not in (K.ALIGN_OK, K.ALIGN_CAPACITY) or (st == K.ALIGN_OK and int(n[b]) != len(ref)):
            # allowed only where the two fp32 sums may truncate differently (and then the test shows that it is so)
            assert _sum_straddles_integer(a, rule), (b, st, int(n[b]), len(ref))
            n_skipped += 1
            continue
        m = min(len(ref), max_frames)
        assert st == (K.ALIGN_OK if len(ref) <= max_frames else K.ALIGN_CAPACITY), (b, st, len(ref))
        assert int(n[b]) == m and at[b, :m].tolist() == ref[:m], b
        assert (at[b, m:] == 0).all(), b
        n_ok += 1
    return n_ok, n_skipped


def _ragged(B, L, seed):
    lens = torch.from_numpy(_rng(seed).integers(0, L + 1, B)).to(torch.int32)
    lens[:3] = torch.tensor([0, 1, L], dtype=torch.int32)
    return lens


# ---------------------------------------------------------------- kernel against host, bit-exact

@pytest.mark.parametrize("kind", ["uniform", "ties", "zeros", "negative"])
def test_rule1_matches_reference_loop(kind):
    B, L = 96, 120
    g = _rng({"uniform": 1, "ties": 2, "zeros": 3, "negative": 4}[kind])
    text = torch.from_numpy(g.integers(1, V, (B, L)))
    a = np.stack([g.random((B, L)), 4.0 * g.random((B, L))], -1).astype(np.float32)
    if kind == "ties":                                     # exact k + 0.5 values: round half to even decides
        a = (np.floor(a * 2) / 2 + 0.5 * (g.random(a.shape) < 0.5)).astype(np.float32)
    elif kind == "zeros":                                  # zero durations and gaps: one-frame minimum, overwrites
        a[g.random(a.shape) < 0.4] = 0.0
    elif kind == "negative":                               # wrap-around indices, non-monotone starts, IndexError
        a = g.normal(0.8, 1.0, a.shape).astype(np.float32)
        a[:8, :3, 0] = -9.0
    text_len = _ragged(B, L, 10)
    n_ok, n_skipped = _check_against_host(text, torch.from_numpy(a), text_len, 1, 4096)
    assert n_ok >= B // 3 and n_skipped <= 2, (n_ok, n_skipped)
    if kind != "negative":                                 # all valid: eager mode against align_batch
        at, n = v.align_frames(text.to(DEV), torch.from_numpy(a).to(DEV), text_len.to(DEV))
        ref, ref_n = v.align_batch(text, torch.from_numpy(a), text_len)
        if torch.equal(n.cpu(), ref_n):
            assert torch.equal(at.cpu(), ref)


def test_golden_align_edges():
    """Every case of the reference-generated align_edges.json: frames where the reference returns, the same exception
    class where it raises, singly and as one ragged batch."""
    with open(os.path.join(GOLDEN, "align_edges.json")) as f:
        cases = json.load(f)
    for c in cases:
        text = torch.tensor([c["text"]], dtype=torch.int64, device=DEV)
        al = torch.tensor([c["align"]], dtype=torch.float32, device=DEV)
        _, _, status = v.align_frames(text, al, max_frames=64)
        if isinstance(c["out"], str):
            assert int(status[0]) in FAILED_AS and FAILED_AS[int(status[0])].__name__ == c["out"], c
            with pytest.raises(FAILED_AS[int(status[0])]):
                v.align_frames(text, al)
            continue
        at, n = v.align_frames(text, al)
        assert int(n[0]) == len(c["out"]) and at[0].tolist() == c["out"], c
    L = max(len(c["text"]) for c in cases)
    text = torch.zeros((len(cases), L), dtype=torch.int64)
    al = torch.full((len(cases), L, 2), 7.0)                # padding past text_len must not be read
    lens = torch.tensor([len(c["text"]) for c in cases], dtype=torch.int32)
    for i, c in enumerate(cases):
        text[i, :len(c["text"])] = torch.tensor(c["text"])
        al[i, :len(c["text"])] = torch.tensor(c["align"])
    at, n, status = v.align_frames(text.to(DEV), al.to(DEV), lens.to(DEV), max_frames=80)
    for i, c in enumerate(cases):
        if isinstance(c["out"], str):
            assert FAILED_AS[int(status[i])].__name__ == c["out"]
        else:
            assert int(status[i]) == K.ALIGN_OK and at[i, :int(n[i])].tolist() == c["out"]


@pytest.mark.parametrize("kind", ["uniform", "short"])
def test_rule2_matches_reference_loop(kind):
    B, L = 80, 90
    g = _rng(20 if kind == "uniform" else 21)
    text = torch.from_numpy(g.integers(1, V, (B, L)))
    a = np.stack([g.random((B, L)), 4.0 * g.random((B, L))], -1).astype(np.float32)
    if kind == "short":                                    # short and zero durations, a few negative entries
        a = (a * 0.3).astype(np.float32)
        a[g.random(a.shape) < 0.3] = 0.0
        a[g.random(a.shape) < 0.05] *= -1.0
    text_len = _ragged(B, L, 11)
    text_len[3:10] = L
    n_ok, n_skipped = _check_against_host(text, torch.from_numpy(a), text_len, 2, 4096)
    assert n_ok >= B - 2 and n_skipped <= 2, (n_ok, n_skipped)
    # align_batch_v2 agrees wherever it does not raise
    for b in range(B):
        n = int(text_len[b])
        try:
            ref, ref_n = v.align_batch_v2(text[b:b + 1, :n], torch.from_numpy(a[b:b + 1, :n]))
        except IndexError:
            continue
        at, at_n = v.align_frames(text[b:b + 1].to(DEV), torch.from_numpy(a[b:b + 1]).to(DEV), text_len[b:b + 1], rule=2)
        if int(at_n[0]) == int(ref_n[0]):
            assert at.cpu()[0, :int(ref_n[0])].tolist() == ref[0, :int(ref_n[0])].tolist(), b


def test_rule2_drops_frames_past_the_total():
    """Known divergence between the two host forms, kept on purpose: with 20 zero-duration tokens every token still
    takes a frame, so the tokens run past head + int(sum) + tail = 10 frames.  TextToAlignText.align (the reference's
    slice assignment) drops the frames past the end and returns 10; align_batch_v2 raises IndexError.  The device
    follows the reference loop."""
    text = torch.arange(1, 21, dtype=torch.int64)[None]
    al = torch.zeros((1, 20, 2))
    ref = v.TextToAlignText.align(text[0], al[0])
    with pytest.raises(IndexError):
        v.align_batch_v2(text, al)
    at, n = v.align_frames(text.to(DEV), al.to(DEV), rule=2)
    assert int(n[0]) == 10 == len(ref) and at[0].tolist() == ref.tolist()


def test_log1p_matches_torch_exp(tts_v1, tts_v2):
    """log1p_input: the durations the kernel works with are bit-equal to torch.exp(pred) - 1 on the same device, for
    the real head outputs of both align models and for fp32 extremes."""
    amodel, _ = tts_v1
    text = torch.from_numpy(synth.text_tokens(16, 100, V, seed=31)).to(DEV)
    preds = [amodel(text)]
    amodel2, _, _ = tts_v2
    lens = torch.full((16,), 100, dtype=torch.int32)
    preds.append(amodel2(text, lens)[0])
    x = torch.linspace(-30.0, 30.0, 16 * 100 * 2, device=DEV).view(16, 100, 2)
    x[0, 0, 0], x[1, 5, 1], x[2, 7, 0], x[3, 9, 1] = -1e30, 1e4, float("nan"), 88.8
    x[4] = torch.randn((100, 2), device=DEV) * 40
    preds.append(x.contiguous())
    for pred in preds:
        d = torch.full(pred.shape, 123.0, device=DEV)
        _, _, status = v.align_frames(text, pred, log1p=True, max_frames=600, durations_out=d)
        ref = torch.exp(pred) - 1
        assert torch.equal(d.view(torch.int32), ref.view(torch.int32)), (d - ref).abs().nan_to_num().max()
    st = status.cpu()
    assert int(st[0]) != K.ALIGN_NAN and int(st[1]) == K.ALIGN_INF and int(st[2]) == K.ALIGN_NAN
    assert (d[0, 0, 0] == -1.0) and math.isinf(float(d[1, 5, 1])) and math.isnan(float(d[2, 7, 0]))
    with pytest.raises(OverflowError):
        v.align_frames(text[1:2], x[1:2].contiguous(), log1p=True)
    with pytest.raises(ValueError):
        v.align_frames(text[2:3], x[2:3].contiguous(), log1p=True)


# ---------------------------------------------------------------- capacity, ownership and layouts

def _direct(align_view, text, text_len, rule, T_cap, sentinel=-777):
    """v100_tts_align called directly into a sentinel-filled output, so that a frame the kernel skips cannot show a
    correct value left by an earlier call."""
    B, L = text.shape
    at = torch.full((B, T_cap), sentinel, dtype=torch.int64, device=DEV)
    out = torch.full((4, B), -5, dtype=torch.int32, device=DEV)
    _lib.call("v100_tts_align", align_view.data_ptr(), *align_view.stride(), 0, None, text.data_ptr(), text.stride(0),
              text_len.data_ptr(), B, L, rule, 5, 5, at.data_ptr(), T_cap, out[0].data_ptr(), out[1].data_ptr(),
              out[2].data_ptr(), out[3].data_ptr(), torch.cuda.current_stream().cuda_stream)
    return at, out


@pytest.mark.parametrize("layout", ["v1_ncw", "v2_tm"])
def test_capacity_sentinel_and_head_layouts(layout):
    """Both head layouts read in place; with a capacity below some totals only those utterances are cut and flagged,
    and every other one is bit-identical to the exact-size result; no sentinel survives in [0, T_cap)."""
    B, L = 45, 100                                          # 45: not a multiple of 8, so Bp > B in the TM layout
    g = _rng(40)
    vals = np.stack([g.random((B, L)), 4.0 * g.random((B, L))], -1).astype(np.float32)
    if layout == "v1_ncw":
        pitch = 104
        data = torch.full((B, 2, pitch), float("nan"))
        data[:, :, :L] = torch.from_numpy(vals).transpose(1, 2)
        data = data.to(DEV)
        view = data.transpose(1, 2)[:, :L]
        assert view.stride() == (2 * pitch, 1, pitch)
    else:
        Bp = 48
        pitch = L * Bp
        data = torch.full((1, 2, pitch), float("nan"))
        tm = data[0].view(2, L, Bp)
        tm[:, :, :B] = torch.from_numpy(vals).permute(2, 1, 0)
        data = data.to(DEV)
        view = torch.as_strided(data, (B, L, 2), (1, Bp, pitch))
    rule = 1 if layout == "v1_ncw" else 2
    text = torch.from_numpy(g.integers(1, V, (B, L))).to(DEV)
    lens = _ragged(B, L, 41).to(DEV)
    full, full_n = v.align_frames(text, torch.from_numpy(vals).to(DEV), lens, rule=rule)
    cap = int(full_n.float().median())
    at, out = _direct(view, text, lens, rule, cap)
    n_total, status, filled, frame_len = out.cpu()
    assert torch.equal(n_total, full_n.cpu())
    cut = full_n.cpu() > cap
    assert cut.any() and (~cut).any()
    assert torch.equal(status, torch.where(cut, K.ALIGN_CAPACITY, K.ALIGN_OK).to(torch.int32))
    assert torch.equal(filled, torch.clamp(full_n.cpu(), max=cap))
    assert torch.equal(frame_len, torch.clamp(2 * filled - 1, min=0))
    assert not (at == -777).any()
    ref = torch.zeros((B, cap), dtype=torch.int64)
    w = min(cap, full.shape[1])
    ref[:, :w] = full.cpu()[:, :w]
    for b in range(B):
        ref[b, int(filled[b]):] = 0
    assert torch.equal(at.cpu(), ref)
    # the wrapper's capacity mode gives the same, from the strided view
    at2, n2, st2 = v.align_frames(text, view, lens, rule=rule, max_frames=cap)
    assert torch.equal(at2, at) and torch.equal(n2.cpu(), filled) and torch.equal(st2.cpu(), status)


def test_plan_only_call_writes_no_frames():
    text = torch.from_numpy(synth.text_tokens(4, 30, V, seed=3)).to(DEV)
    al = torch.from_numpy(synth.synthetic_alignment(4, 30, seed=3)).to(DEV)
    at, out = K.tts_align(text, al, None, 1, 5, 5, None, False)
    ref, ref_n = v.align_batch(text.cpu(), al.cpu())
    assert at is None and torch.equal(out[0].cpu(), ref_n) and (out[1] == 0).all()


def test_too_many_tokens_is_unsupported():
    text = torch.ones((1, 4097), dtype=torch.int64, device=DEV)
    with pytest.raises(_lib.V100Error, match="4096"):
        v.align_frames(text, torch.zeros((1, 4097, 2), device=DEV), max_frames=8)


# ---------------------------------------------------------------- pipelines

def _load(model, sd):
    model.load_state_dict({k: torch.from_numpy(np.asarray(t)) for k, t in sd.items()})
    return model.to(DEV).eval()


def _realistic_head(sd, key, scale=0.1):
    """Head weights scaled down and biases log1p((0.5, 2.0)): about 2.5 frames a token, as trained models give."""
    sd = dict(sd)
    sd[key + ".weight"] = (np.asarray(sd[key + ".weight"]) * scale).astype(np.float32)
    sd[key + ".bias"] = np.log1p(np.array([0.5, 2.0], np.float32)).astype(np.float32)
    return sd


@pytest.fixture(scope="module")
def tts_v1():
    H = 512
    amodel = _load(v.TextToAlignTextModel(V, H), _realistic_head(synth.align_state_dict(V, H, seed=61), "layers.4"))
    vmodel = _load(v.AlignTextToAudioModel(V, H), synth.audio_state_dict(V, H, seed=61, randomize_norm=True))
    return amodel, vmodel


@pytest.fixture(scope="module")
def tts_v2():
    amodel = _load(v.TextToAlignText(V, 2, 256, 2), _realistic_head(synth.align_v2_state_dict(V, 2, 256, 2, seed=62),
                                                                    "dense"))
    dec = [list(r) for r in synth.TTS_V2_BASE_DECODER]
    vmodel = _load(v.AlignTextToAudio(V, 257, 1, 2, 512, dec), synth.audio_v2_state_dict(V, seed=62, randomize_norm=True))
    mcep = _load(v.AlignTextToAudio(V, 25, 1, 2, 512, dec), synth.audio_v2_state_dict(V, 25, seed=63,
                                                                                     randomize_norm=True))
    return amodel, vmodel, v.AlignTextToAudioPredict(mcep).to(DEV)


def _same(a, b):
    return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


def _stepwise_v1(amodel, vmodel, text, text_len):
    pred = amodel(text.to(DEV))
    align = torch.exp(pred) - 1
    at, at_len = v.align_batch(text.cpu(), align.cpu(), text_len)
    return vmodel.predict(at.to(DEV)), at_len, align


def test_tts_pipeline_matches_stepwise(tts_v1):
    """BASELINE configs[2] shape (tts_en_base, 256 x 100 tokens, ragged text_len): the pipeline is bit-identical to
    align model -> torch.exp - 1 -> align_batch -> predict."""
    amodel, vmodel = tts_v1
    B, L = 256, 100
    text = torch.from_numpy(synth.text_tokens(B, L, V, seed=71))
    text_len = torch.from_numpy(_rng(72).integers(60, L + 1, B)).to(torch.int32)
    (f0, logspc, codeap), at_len, _ = _stepwise_v1(amodel, vmodel, text, text_len)
    assert 150 < float(at_len.float().mean()) < 350                                   # about 2.5 frames a token
    got = v.TtsPipeline(amodel, vmodel)(text.to(DEV), text_len.to(DEV))
    assert _same(got[0], f0) and _same(got[1], logspc) and _same(got[2], codeap)
    assert torch.equal(got[3].cpu(), 2 * at_len - 1) and (got[4] == 0).all()


def test_tts_pipeline_random_init_negative_durations():
    """Random-init head weights (only the bias set to log1p((0.5, 2.0)), so that the totals stay positive and no
    token runs past the end) predict negative gaps and durations for about a quarter of the entries: non-monotone
    starts and overwritten frames run end to end, and the result still matches the stepwise composition, whose
    align_batch takes the reference's per-utterance loop for such utterances.  (With the bias left random, most of
    these utterances sum to a negative duration and the reference itself raises; wrap-around indices are covered by
    the kernel tests above.)"""
    H = 512
    sd = dict(synth.align_state_dict(V, H, seed=81))
    sd["layers.4.bias"] = np.log1p(np.array([0.5, 2.0], np.float32))
    amodel = _load(v.TextToAlignTextModel(V, H), sd)
    vmodel = _load(v.AlignTextToAudioModel(V, H), synth.audio_state_dict(V, H, seed=81))
    text = torch.from_numpy(synth.text_tokens(8, 40, V, seed=82))
    (f0, logspc, codeap), at_len, align = _stepwise_v1(amodel, vmodel, text, None)
    assert (align[..., 0] < 0).sum() > 40 and (align[..., 1] < 0).any()
    got = v.TtsPipeline(amodel, vmodel)(text.to(DEV))
    assert _same(got[0], f0) and _same(got[1], logspc) and _same(got[2], codeap)
    assert torch.equal(got[3].cpu(), 2 * at_len - 1)


@pytest.mark.parametrize("which", ["AlignTextToAudio", "AlignTextToAudioPredict"])
def test_tts_v2_pipeline_matches_stepwise(tts_v2, which):
    amodel, vmodel, wrapped = tts_v2
    audio = vmodel if which == "AlignTextToAudio" else wrapped
    B, L = 64, 100
    text = torch.from_numpy(synth.text_tokens(B, L, V, seed=91))
    text_len = torch.from_numpy(_rng(92).integers(1, L + 1, B)).to(torch.int32)
    text_len[0] = L
    align, _ = amodel.predict(text.to(DEV), text_len)
    at, at_len = v.align_batch_v2(text, align.cpu(), text_len)
    ref = audio.predict(at.to(DEV), at_len) if which == "AlignTextToAudio" else audio(at.to(DEV), at_len)
    got = v.TtsV2Pipeline(amodel, audio)(text.to(DEV), text_len.to(DEV))
    for g_, r_ in zip(got[:3], ref):
        assert _same(g_, r_)
    assert torch.equal(got[3].cpu(), 2 * at_len - 1) and (got[4] == 0).all()


@pytest.mark.parametrize("version", [1, 2])
def test_graphed_matches_eager(tts_v1, tts_v2, version):
    """One CUDA graph for text -> WORLD parameters; two replays with different texts each equal their own eager
    result at the same max_frames, bit for bit."""
    if version == 1:
        pipe, max_frames = v.TtsPipeline(*tts_v1), 240
    else:
        pipe, max_frames = v.TtsV2Pipeline(tts_v2[0], tts_v2[1]), 200
    B, L = 24, 80
    run = pipe.graphed(B, L, max_frames)
    for seed in (101, 102):
        text = torch.from_numpy(synth.text_tokens(B, L, V, seed=seed)).to(DEV)
        text_len = torch.from_numpy(_rng(seed).integers(1, L + 1, B)).to(torch.int32).to(DEV)
        got = [t.clone() for t in run(text, text_len)]
        ref = pipe(text, text_len, max_frames)
        for g_, r_ in zip(got[:3], ref[:3]):
            assert _same(g_, r_)
        assert torch.equal(got[3], ref[3]) and torch.equal(got[4], ref[4])
        assert int(got[0].shape[1]) == 2 * max_frames - 1
