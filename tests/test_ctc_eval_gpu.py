"""ASR evaluation on the device: v100_ctc_loss against torch's own ctc_loss in float64 on the CPU, v100_edit_distance
against a plain DP (exactly), and AsrPipeline / AsrV2Pipeline.evaluate against the pieces it is made of."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import voice100_b200 as v
from voice100_b200 import kernels as K, v2
from ctc_eval_reference import edit_distance_np
from helpers import asr_case, asr_v2_case

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _logits(T, B, V, peaked, seed):
    g = torch.Generator().manual_seed(seed)
    return (8.0 if peaked else 0.01) * torch.randn(T, B, V, generator=g)


def _batch(T, B, V, L, seed, blank=0):
    """Ragged lengths with 0 and T among the inputs and 0 and L among the targets; labels drawn from all of [0, V),
    so some equal `blank`; rows 4-6 repeat one label, which forces a blank between every pair of them: row 4 has
    exactly enough frames, row 5 one too few."""
    rng = np.random.default_rng(seed)
    il = rng.integers(0, T + 1, B)
    tl = rng.integers(0, L + 1, B)
    il[0], il[1], tl[2], tl[3] = 0, T, 0, L
    tl[0] = 0                                          # input 0, target 0: loss 0
    tg = rng.integers(0, V, (B, L))
    n_rep = min(L, (T + 1) // 2)
    lab = (blank + 1) % V
    tg[4:7, :] = lab
    tl[4:7] = n_rep
    il[4], il[5], il[6] = 2 * n_rep - 1, 2 * n_rep - 2, T
    il[7], tl[7] = 3, 5                                # too few frames for the target
    return torch.from_numpy(tg), torch.from_numpy(il), torch.from_numpy(tl)


def _ref(x, targets, il, tl, blank=0, normalize=False, zero_infinity=False):
    lp = x.double().cpu()
    if normalize:
        lp = lp.log_softmax(-1)
    return F.ctc_loss(lp, targets.cpu(), il.cpu(), tl.cpu(), blank=blank, reduction="none",
                      zero_infinity=zero_infinity)


def _check(got, ref):
    got = got.cpu().double()
    assert torch.equal(torch.isinf(got), torch.isinf(ref)), (torch.isinf(got) != torch.isinf(ref)).nonzero()
    assert not torch.isnan(got).any()
    fin = torch.isfinite(ref)
    err = (got[fin] - ref[fin]).abs() / ref[fin].abs().clamp_min(1)
    assert float(err.max()) <= 1e-6, float(err.max())
    return int((~fin).sum())


@pytest.mark.parametrize("V", [29, 44, 71])
@pytest.mark.parametrize("peaked", [True, False])
@pytest.mark.parametrize("normalize", [True, False])
def test_ctc_loss_matches_torch_float64(V, peaked, normalize):
    T, B, L = 751, 256, 300
    x = _logits(T, B, V, peaked, seed=V + 2 * peaked)
    if not normalize:
        x = x.log_softmax(-1)
    tg, il, tl = _batch(T, B, V, L, seed=V)
    got = v.ctc_loss(x.to(DEV), tg.to(DEV), il.to(DEV), tl.to(DEV), reduction="none", normalize=normalize)
    n_inf = _check(got, _ref(x, tg, il, tl, normalize=normalize))
    assert n_inf >= 2 and float(got[0]) == 0.0
    # zero_infinity: the same values with every inf replaced by exactly 0
    gz = v.ctc_loss(x.to(DEV), tg.to(DEV), il.to(DEV), tl.to(DEV), reduction="none", normalize=normalize,
                    zero_infinity=True)
    assert torch.equal(gz, torch.where(torch.isinf(got), torch.zeros_like(got), got))
    # host-resident lengths: the same launch after the host checks
    gh = v.ctc_loss(x.to(DEV), tg.to(DEV), il.tolist(), tl, reduction="none", normalize=normalize)
    assert torch.equal(gh, got)


def test_ctc_loss_blank_last_and_concatenated_targets():
    T, B, V, L = 400, 64, 44, 120
    x = _logits(T, B, V, True, seed=1).log_softmax(-1)
    tg, il, tl = _batch(T, B, V, L, seed=2, blank=V - 1)
    ref = _ref(x, tg, il, tl, blank=V - 1)
    got = v.ctc_loss(x.to(DEV), tg.to(DEV), il.to(DEV), tl.to(DEV), blank=V - 1, reduction="none")
    _check(got, ref)
    flat = torch.cat([tg[b, :int(tl[b])] for b in range(B)])
    assert torch.equal(_ref(x, flat, il, tl, blank=V - 1), ref)
    for lengths in ((il.to(DEV), tl.to(DEV)), (il.tolist(), tl.tolist())):      # device offsets / host offsets
        got1 = v.ctc_loss(x.to(DEV), flat.to(DEV), *lengths, blank=V - 1, reduction="none")
        assert torch.equal(got1, got)
    # int32 lengths and int32 targets are accepted as torch accepts them
    got2 = v.ctc_loss(x.to(DEV), tg.to(DEV, torch.int32), il.to(DEV, torch.int32), tl.to(DEV, torch.int32),
                      blank=V - 1, reduction="none")
    assert torch.equal(got2, got)


def test_ctc_loss_reads_v1_and_v2_layouts_in_place():
    T, B, V, L = 300, 40, 29, 80
    tg, il, tl = _batch(T, B, V, L, seed=3)
    x = _logits(T, B, V, True, seed=3)
    ref = _ref(x, tg, il, tl, normalize=True)
    args = (tg.to(DEV), il.to(DEV), tl.to(DEV))
    dense = v.ctc_loss(x.to(DEV).contiguous(), *args, reduction="none", normalize=True)
    _check(dense, ref)
    v1 = x.transpose(0, 1).contiguous().to(DEV)                     # [B, T, V]: the v1 head's logits
    view = v1.transpose(0, 1)
    assert view.stride() == (V, T * V, 1)
    assert torch.equal(v.ctc_loss(view, *args, reduction="none", normalize=True), dense)
    tm = torch.randn(T, 48, V, device=DEV)                          # [T, Bp, V]: the v2 head's time-major logits
    tm[:, :B] = x.to(DEV)
    assert torch.equal(v.ctc_loss(tm[:, :B], *args, reduction="none", normalize=True), dense)


def test_ctc_loss_long_utterance():
    T, B, V, L = 3001, 4, 71, 900
    x = _logits(T, B, V, True, seed=4)
    rng = np.random.default_rng(4)
    tg = torch.from_numpy(rng.integers(1, V, (B, L)))
    il = torch.tensor([3001, 3001, 2500, 1801])
    tl = torch.tensor([900, 450, 900, 900])
    tg[3, :] = 7                                                    # 900 repeats need 1799 frames: 1801 suffice
    got = v.ctc_loss(x.to(DEV), tg.to(DEV), il.to(DEV), tl.to(DEV), reduction="none", normalize=True)
    assert _check(got, _ref(x, tg, il, tl, normalize=True)) == 0


def test_ctc_loss_reductions_match_torch_expression():
    T, B, V, L = 200, 32, 29, 60
    x = _logits(T, B, V, True, seed=5).log_softmax(-1).to(DEV)
    tg, il, tl = _batch(T, B, V, L, seed=5)
    tg, il, tl = tg.to(DEV), il.to(DEV), tl.to(DEV)
    none = v.ctc_loss(x, tg, il, tl, reduction="none", zero_infinity=True)
    assert torch.equal(v.ctc_loss(x, tg, il, tl, reduction="sum", zero_infinity=True), none.sum())
    assert torch.equal(v.ctc_loss(x, tg, il, tl, zero_infinity=True),
                       (none / tl.to(none.dtype).clamp_min(1)).mean())


def test_ctc_loss_statuses_and_isolation():
    T, B, V, L = 120, 12, 29, 30
    x = _logits(T, B, V, True, seed=6).log_softmax(-1).to(DEV)
    tg, il, tl = _batch(T, B, V, L, seed=6)
    tg, il, tl = tg.to(DEV), il.to(DEV), tl.to(DEV)
    clean, st, _ = K.ctc_loss_batch(x, tg, il, tl)
    assert st.tolist() == [K.CTC_OK] * B
    tg2, il2, tl2 = tg.clone(), il.clone(), tl.clone()
    tl2[8], tl2[9] = 10, 10
    tg2[8, 3], tg2[9, 9], tg2[9, 10] = V, -1, V + 5                # out-of-range labels inside the target
    tg2[10, int(tl[10]):] = -7                                     # out of range, but past the length: ignored
    il2[1], il2[2], tl2[3] = T + 1, -1, L + 1                       # lengths outside [0, T] / [0, width]
    loss, st, _ = K.ctc_loss_batch(x, tg2, il2, tl2)
    st = st.tolist()
    assert st[8] == st[9] == K.CTC_BAD_LABEL and st[1] == st[2] == st[3] == K.CTC_BAD_LENGTH
    bad = [1, 2, 3, 8, 9]
    assert torch.isnan(loss[bad]).all()
    keep = [b for b in range(B) if b not in bad]
    assert all(st[b] == K.CTC_OK for b in keep) and torch.equal(loss[keep], clean[keep])
    # concatenated targets whose lengths run past the buffer
    flat = torch.cat([tg[b, :int(tl[b])] for b in range(B)])
    tl3 = tl.clone()
    tl3[B - 1] += 1
    loss3, st3, _ = K.ctc_loss_batch(x, flat, il, tl3)
    assert st3.tolist()[-1] == K.CTC_BAD_LENGTH and torch.equal(loss3[:-1], clean[:-1])
    # device lengths with a padded width above the limit: unsupported, not a silent fallback
    wide = torch.zeros(B, K.CTC_MAX_TARGET + 1, dtype=torch.int64, device=DEV)
    with pytest.raises(v.V100Error, match="limit"):
        v.ctc_loss(x, wide, il, tl)


def test_ctc_loss_deterministic_and_batch_independent():
    T, B, V, L = 751, 64, 44, 200
    x = _logits(T, B, V, False, seed=7).to(DEV)
    tg, il, tl = _batch(T, B, V, L, seed=7)
    tg, il, tl = tg.to(DEV), il.to(DEV), tl.to(DEV)
    runs = [v.ctc_loss(x, tg, il, tl, reduction="none", normalize=True) for _ in range(3)]
    assert all(torch.equal(r, runs[0]) for r in runs)
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(0)).to(DEV)[: B // 3]
    sub = v.ctc_loss(x[:, perm].contiguous(), tg[perm], il[perm], tl[perm], reduction="none", normalize=True)
    assert torch.equal(sub, runs[0][perm])


def _pairs(B, Lh, Lr, alphabet, seed, base=0):
    rng = np.random.default_rng(seed)
    hyp = base + rng.integers(0, alphabet, (B, Lh))
    ref = base + rng.integers(0, alphabet, (B, Lr))
    hl = rng.integers(0, Lh + 1, B)
    rl = rng.integers(0, Lr + 1, B)
    hl[0], rl[0] = Lh, Lr
    return hyp, hl, ref, rl


def _dev(*arrs):
    return [torch.from_numpy(np.asarray(a)).to(DEV) for a in arrs]


@pytest.mark.parametrize("alphabet,base", [(2, 0), (29, 0), (71, 0), (5, (1 << 40) - 2)])
def test_edit_distance_matches_dp(alphabet, base):
    B, Lh, Lr = 96, 150, 170
    hyp, hl, ref, rl = _pairs(B, Lh, Lr, alphabet, seed=alphabet, base=base)
    hyp[1], hl[1], rl[1] = ref[1, :Lh], min(Lh, rl[1]), min(Lh, rl[1])   # identical
    hyp[2] = base + alphabet + 3                                          # disjoint from every id of its reference
    hl[3], rl[4], hl[5], rl[5] = 0, 0, 0, 0                               # empty on one side, on both
    got = v.edit_distance(*_dev(hyp), *_dev(hl), *_dev(ref), *_dev(rl)).cpu().tolist()
    want = [edit_distance_np(hyp[b, :hl[b]], ref[b, :rl[b]]) for b in range(B)]
    assert got == want
    assert got[1] == 0 and got[2] == max(hl[2], rl[2]) and got[3] == rl[3] and got[5] == 0


def test_edit_distance_lengths():
    sizes = [63, 64, 65, 127, 128, 129, 2048]
    rng = np.random.default_rng(9)
    pairs = [(a, b) for a in sizes for b in (sizes[0], sizes[4], 2048)] + [(16384, 2048), (2048, 16384),
                                                                             (16384, 16384), (16384, 0)]
    W = 16384
    hyp = np.zeros((len(pairs), W), np.int64)
    ref = np.zeros((len(pairs), W), np.int64)
    for k, (a, b) in enumerate(pairs):
        base = rng.integers(0, 29, max(a, b))
        hyp[k, :a] = base[:a]
        r = base[:b].copy()
        flip = rng.random(b) < 0.3
        r[flip] = rng.integers(0, 29, int(flip.sum()))
        ref[k, :b] = r
    hl = np.array([a for a, _ in pairs])
    rl = np.array([b for _, b in pairs])
    got = v.edit_distance(*_dev(hyp), *_dev(hl), *_dev(ref), *_dev(rl)).cpu().tolist()
    want = [edit_distance_np(hyp[k, :a], ref[k, :b]) for k, (a, b) in enumerate(pairs)]
    assert got == want
    # device lengths beyond the padded width are clamped to it, negative ones to 0 (as ctc_collapse does)
    h, r = _dev(hyp[:3, :100], ref[:3, :90])
    got = v.edit_distance(h, torch.tensor([500, -4, 50], device=DEV), r, torch.tensor([90, 30, 10 ** 6], device=DEV))
    assert got.tolist() == [edit_distance_np(hyp[0, :100], ref[0, :90]), 30,
                            edit_distance_np(hyp[2, :50], ref[2, :90])]
    with pytest.raises(v.V100Error):
        v.edit_distance(torch.zeros(1, W + 1, dtype=torch.int64, device=DEV), None, r[:1], None)


def _texts(B, V, out_len, seed):
    """Seeded transcripts of about a third of each utterance's frames; the shortest utterance gets one as long as the
    longest, which is too long for it (zero_infinity turns its inf into 0)."""
    rng = np.random.default_rng(seed)
    ol = out_len.cpu().numpy()
    S = int(ol.max())
    n = np.minimum(rng.integers(1, np.maximum(ol // 3, 2)), S)
    n[int(ol.argmin())] = S
    text = rng.integers(1, V, (B, S))
    return torch.from_numpy(text).to(DEV), torch.from_numpy(n).to(DEV)


def _check_evaluate(pipe, wav, lens, logits_tbv, x_len, V):
    tokens_ids = pipe.transcribe_ids(wav, lens)
    text, tlen = _texts(wav.shape[0], V, x_len, seed=11)
    loss, errors, ids, counts = pipe.evaluate(wav, lens, text, tlen)
    assert torch.equal(ids, tokens_ids[0]) and torch.equal(counts, tokens_ids[1])
    ref_loss = v.ctc_loss(logits_tbv, text, x_len, tlen, reduction="none", zero_infinity=True, normalize=True)
    assert torch.equal(loss, ref_loss)
    ids_c, cnt_c, text_c, tlen_c = ids.cpu(), counts.cpu(), text.cpu(), tlen.cpu()
    want = [edit_distance_np(ids_c[b, :cnt_c[b]].numpy(), text_c[b, :tlen_c[b]].numpy()) for b in range(len(cnt_c))]
    assert errors.cpu().tolist() == want
    # the float64 oracle on the same logits
    _check(loss, _ref(logits_tbv.cpu(), text_c, x_len.cpu(), tlen_c, normalize=True, zero_infinity=True))
    # three repeated calls are bit-identical
    for _ in range(2):
        again = pipe.evaluate(wav, lens, text, tlen)
        assert all(torch.equal(a, b) for a, b in zip(again, (loss, errors, ids, counts)))
    # an utterance's loss does not depend on the rest of the batch
    perm = torch.tensor([2, 0], device=DEV)
    sub = v.ctc_loss(logits_tbv[:, perm].contiguous(), text[perm], x_len[perm], tlen[perm], reduction="none",
                     zero_infinity=True, normalize=True)
    assert torch.equal(sub, loss[perm])
    # a CUDA-graph capture of evaluate replays to the same bits
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        pipe.evaluate(wav, lens, text, tlen)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = pipe.evaluate(wav, lens, text, tlen)
    graph.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(static, (loss, errors, ids, counts)))
    return loss


def test_asr_v1_evaluate():
    sd, wav, lengths, g = asr_case("asr_ja_phone_ragged")
    audio_size, embed, vocab, hidden = [int(x) for x in g["cfg"][:4]]
    model = v.AudioToTextCTC(audio_size, embed, vocab, hidden)
    model.load_state_dict(sd)
    model = model.to(DEV).eval()
    tr = v.MelSpectrogramAudioTransform().to(DEV)
    pipe = v.AsrPipeline(tr, model)
    wav, lens = wav.to(DEV), torch.tensor(lengths, dtype=torch.int32, device=DEV)
    with torch.no_grad():
        feats, audio_len = tr.logmel_batch(wav, lens, ncw_dtype=model.storage_dtype)
        logits, _, out_len = model._run(feats, True, audio_len)
    n0 = v._lib.stats["launches"]
    pipe(wav, lens)
    n1 = v._lib.stats["launches"]
    pipe.evaluate(wav, lens, *_texts(wav.shape[0], vocab, out_len, seed=11))
    assert v._lib.stats["launches"] - n1 == (n1 - n0) + 3 == 33     # __call__'s 30, then loss, collapse, distance
    _check_evaluate(pipe, wav, lens, logits.transpose(0, 1), out_len, vocab)


def test_asr_v2_evaluate():
    sd, wav, lengths, settings, g = asr_v2_case("asr_v2_en_small_ragged")
    audio_size, hidden, vocab = [int(x) for x in g["cfg"][:3]]
    model = v2.AudioToAlignText(audio_size, [list(r) for r in settings], 2, hidden, vocab)
    model.load_state_dict(sd, strict=False)
    model = model.to(DEV).eval()
    tr = v.MelSpectrogramAudioTransform().to(DEV)
    pipe = v2.AsrV2Pipeline(tr, model)
    wav, lens = wav.to(DEV), torch.tensor(lengths, dtype=torch.int32, device=DEV)
    with torch.no_grad():
        feats, audio_len = tr.logmel_batch(wav, lens, ncw_dtype=model.storage_dtype)
        x_len = model.output_length(audio_len)
        y, tm = model._run(feats, x_len)
        logits = K.ctc_finalize(y, want_logits=True)[0].view(tm.T, tm.Bp, vocab)[:, :tm.B]
    _check_evaluate(pipe, wav, lens, logits, x_len, vocab)
