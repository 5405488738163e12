"""Every libv100 entry point once, at small shapes, for compute-sanitizer (memcheck / racecheck / synccheck):
    compute-sanitizer --tool memcheck python tools/sanitize_small.py
"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
import voice100_b200 as v
from voice100_b200 import kernels as K, synth
dev = "cuda"
torch.manual_seed(0)
MODE = os.environ.get("SAN_MODE", "all")   # all | nogemm (everything that does not use TMA/mbarrier/tcgen05) | v2
if MODE == "v2":
    # the v2 kernels: tap stack + GEMM, LayerNorm/GELU, layout changes, the LSTM pair kernel (ragged, 2 groups)
    m = v.AudioToAlignText(64, [[128, False, 3, 2, 1, False], [128, False, 5, 1, 2, True]], 2, 128, 29).to(dev).eval()
    B = 70
    audio = torch.randn(B, 37, 64, device=dev)
    audio_len = torch.randint(1, 38, (B,), device=dev)
    audio_len[0] = 37
    for dtype in (torch.bfloat16, torch.float16):
        m.set_storage_dtype(dtype)
        logits, lens = m(audio, audio_len)
        tok, _ = m.greedy(audio, audio_len)
    al = v.TextToAlignText(29, 2, 64, 2).to(dev).eval()
    al(torch.randint(1, 29, (3, 11), device=dev), torch.tensor([11, 4, 7]))
    tts = v.AlignTextToAudio(29, 25, 1, 2, 64, [[64, False, 5, 1, 2, False], [64, True, 5, 2, 2, False], [64, False, 5, 1, 2, False]]).to(dev).eval()
    tts.predict(torch.randint(1, 29, (3, 21), device=dev), torch.tensor([21, 9, 14]))
    v.AlignTextToAudioPredict(tts).to(dev)(torch.randint(1, 29, (3, 21), device=dev), torch.tensor([21, 9, 14]))
    torch.cuda.synchronize()
    print("sanitize_small (v2) done")
    sys.exit(0)
if MODE == "nogemm":
    tr = v.MelSpectrogramAudioTransform().to(dev)
    wav = 0.1 * torch.randn(3, 16000 * 2 + 123, device=dev)
    ln = torch.tensor([32123, 9000, 20001], dtype=torch.int32, device=dev)
    tr.logmel_batch(wav, ln); tr.logmel_batch(wav, ln, ncw_dtype=torch.float16); tr.melspec(wav[0])
    pcm = (wav * 32767).to(torch.int16)
    tr.logmel_batch(pcm, ln, ncw_dtype=torch.bfloat16); tr.logmel_batch(pcm[:, :32001].contiguous(), ln.clamp(max=32001))
    tr.logmel_batch(wav, torch.tensor([0, 1, 10 ** 6], dtype=torch.int32, device=dev))      # empty / too short / over-long
    for dtype in (torch.bfloat16, torch.float16):
        x = K.empty_ncw(2, 72, 333, dev, dtype); x.data.normal_()
        for k in (5, 11, 35, 83):
            w = torch.randn(72, k, device=dev).to(dtype)
            for simt in (False, True):
                K.dwconv(x, w, None, torch.zeros(72, device=dev), k, 1, 1, simt=simt)
            K.dwconv(x, w, None, torch.zeros(72, device=dev), k, 2, 1)
        K.ncw_to_f32(K.ncw_from_f32(torch.randn(2, 7, 33, device=dev), dtype))
        K.ntc_f32_to_ncw(torch.randn(2, 33, 64, device=dev), dtype)
        K.embedding_ncw(torch.randint(0, 29, (2, 19), device=dev), torch.randn(29, 64, device=dev).to(dtype))
    lg = K.Ncw(torch.randn(2, 29, 56, device=dev), 51)
    _, tok = K.ctc_finalize(lg)
    K.ctc_collapse(tok, torch.tensor([51, 20], device=dev))
    K.ncw_f32_to_ntc(lg)
    K.world_finalize(K.Ncw(torch.randn(2, 260, 56, device=dev), 53), torch.zeros(259, device=dev), torch.ones(259, device=dev), True)
    K.world_finalize(K.Ncw(torch.randn(2, 33, 56, device=dev), 53), torch.zeros(29, device=dev), torch.ones(29, device=dev), True, 25, 3, 2)
    _, _, ol = K.ctc_finalize(lg, False, torch.tensor([51, 20], dtype=torch.int32, device=dev))
    lp = torch.log_softmax(torch.randn(3, 50, 29, device=dev), -1)
    v.ctc_best_path_batch(lp, torch.tensor([50, 30, 4]), torch.randint(1, 29, (3, 9), device=dev), torch.tensor([9, 5, 9]))
    v.ctc_best_path_batch(lp * 3, torch.tensor([50, 9, 4]), torch.randint(1, 29, (3, 9), device=dev), torch.tensor([9, 9, 0]), normalize=True)
    torch.cuda.synchronize()
    print("sanitize_small (nogemm) done")
    sys.exit(0)
for dtype in (torch.bfloat16, torch.float16):
    asr = v.AudioToTextCTC(64, 64, 29, 64)
    asr.load_state_dict({k: torch.from_numpy(np.asarray(t)) for k, t in synth.asr_state_dict(64, 64, 29, 64, seed=1, randomize_bn=True).items()})
    asr = asr.to(dev).eval().set_storage_dtype(dtype)
    pipe = v.AsrPipeline(v.MelSpectrogramAudioTransform().to(dev), asr)
    wav = 0.1 * torch.randn(3, 16000 * 2 + 123, device=dev)
    ln = torch.tensor([32123, 9000, 20001], dtype=torch.int32, device=dev)
    tok, out_len = pipe(wav, ln)
    ids, counts = pipe.transcribe_ids(wav, ln)
    audio, _ = pipe.transform.logmel_batch(wav, ln)
    logits = asr(audio)
    asr.encoder(audio.transpose(1, 2).contiguous())
    pipe.transform.melspec(wav[0])
    al = v.TextToAlignTextModel(29, 64).to(dev).eval().set_storage_dtype(dtype)
    au = v.AlignTextToAudioModel(29, 64).to(dev).eval().set_storage_dtype(dtype)
    text = torch.randint(1, 29, (2, 21), device=dev)
    al(text)
    au.predict(torch.randint(0, 29, (2, 45), device=dev))
    # odd shapes straight through the kernels
    x = K.empty_ncw(2, 72, 333, dev, dtype); x.data.normal_()
    W = torch.randn(200, 72, device=dev).to(dtype)
    K.conv1x1(x, W, torch.rand(200, device=dev), torch.zeros(200, device=dev), 1)
    K.conv1x1_f32(x, W[:29].contiguous(), torch.zeros(29, device=dev))
    w = torch.randn(72, 83, device=dev).to(dtype)
    for simt in (False, True):
        K.dwconv(x, w, None, torch.zeros(72, device=dev), 83, 1, 1, simt=simt)
    K.dwconv(x, w[:, :11].contiguous(), None, torch.zeros(72, device=dev), 11, 2, 1)
    # weights-resident pair GEMM (needs >= 4 units per pair slot: 40 utterances x 2 time tiles, 4 channel blocks), with and
    # without a residual; bulk-staged depthwise at odd lengths (T & 7 != 0, several chunks, fewer than 8 samples)
    xw = K.empty_ncw(40, 256, 140, dev, dtype); xw.data.normal_()
    Ww = torch.randn(1024, 256, device=dev).to(dtype) / 16
    yw = K.conv1x1(xw, Ww, torch.rand(1024, device=dev), torch.zeros(1024, device=dev), 1)
    K.conv1x1(yw, torch.randn(256, 1024, device=dev).to(dtype) / 32, None, torch.zeros(256, device=dev), 0, xw)
    for (Tb, kb) in ((1027, 35), (5, 19), (2049, 59)):
        xb = K.empty_ncw(3, 16, Tb, dev, dtype); xb.data.normal_()
        K.dwconv(xb, torch.randn(16, kb, device=dev).to(dtype), None, torch.zeros(16, device=dev), kb, 1, 1)
lp = torch.log_softmax(torch.randn(3, 50, 29, device=dev), -1)
v.ctc_best_path_batch(lp, torch.tensor([50, 30, 4]), torch.randint(1, 29, (3, 9), device=dev), torch.tensor([9, 5, 9]))
torch.cuda.synchronize()
print("sanitize_small done")
