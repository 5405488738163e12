"""CPU-side checks of the drop-in boundary: libv100.so loads without a GPU and exports exactly the
symbols include/v100.h declares; the ctypes table matches the header; product code never imports the
oracle; modules refuse to run without CUDA."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest
import torch

import voice100_b200 as v
from voice100_b200 import _lib, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "v100.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    decls = re.findall(r"\b(?:int|int64_t|const char\*)\s+(v100_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S)
    return {name: [a.strip() for a in args.split(",")] if args.strip() != "void" else [] for name, args in decls}


def test_library_loads_and_exports_header_symbols():
    from voice100_b200 import build
    build.build()
    assert os.path.exists(_lib.LIB_PATH)
    handle = ctypes.CDLL(_lib.LIB_PATH)
    funcs = header_functions()
    assert len(funcs) >= 15
    for name in funcs:
        assert hasattr(handle, name), f"{name} declared in v100.h but not exported"
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (v100_\w+)", out))
    assert exported == set(funcs), exported ^ set(funcs)
    assert _lib.lib().v100_abi_version() == _lib.ABI_VERSION == 8


def test_plain_c_consumer_compiles_links_and_fails_loudly(tmp_path):
    """include/v100.h is a C header: a C99 translation unit (what a cgo / JNI / FFI binding compiles) must build against it
    with no CUDA or C++ headers, link to libv100.so, see the header's ABI version, and get an ERROR (not a host fallback)
    from a compute entry point on a box without a GPU."""
    from voice100_b200 import build
    build.build()
    exe = str(tmp_path / "consumer")
    libdir = os.path.dirname(_lib.LIB_PATH)
    cmd = ["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "c", "consumer.c"), "-o", exe, "-L", libdir, "-l:" + os.path.basename(_lib.LIB_PATH),
           "-Wl,-rpath," + libdir]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    assert "conv1x1(NULL...) -> -1" in r.stdout, r.stdout


def test_ctypes_table_matches_header():
    funcs = header_functions()
    for name, argtypes in _lib.SIGNATURES.items():
        assert name in funcs, name
        assert len(argtypes) == len(funcs[name]), (name, len(argtypes), funcs[name])
        for ct, decl in zip(argtypes, funcs[name]):
            if "*" in decl:
                assert ct is ctypes.c_void_p, (name, decl)
            elif decl.startswith("int64_t"):
                assert ct is ctypes.c_int64, (name, decl)
            elif decl.startswith("float"):
                assert ct is ctypes.c_float, (name, decl)
            else:
                assert ct is ctypes.c_int, (name, decl)
    assert set(funcs) - set(_lib.SIGNATURES) == {"v100_last_error", "v100_lstm_workspace_bytes"}


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "voice100_b200")):
        for f in files:
            if f.endswith(".py"):
                text = open(os.path.join(dirpath, f)).read()
                assert "v100_oracle" not in text and "import oracle" not in text, f


def test_no_cpu_fallback():
    m = v.AudioToTextCTC(64, 128, 29, 128)
    with pytest.raises(v.V100Error):
        m(torch.zeros(1, 50, 64))
    with pytest.raises(v.V100Error):
        v.MelSpectrogramAudioTransform().melspec(torch.zeros(1000))
    with pytest.raises(v.V100Error):
        v.TextToAlignTextModel(29, 64)(torch.zeros(1, 5, dtype=torch.long))
    with pytest.raises(v.V100Error):
        v.AudioToAlignText(64, [list(r) for r in synth.ASR_V2_SMALL_ENCODER], 2, 256, 29)(
            torch.zeros(1, 50, 64), torch.tensor([50]))
    with pytest.raises(v.V100Error):
        v.TextToAlignText(29, 2, 64, 2)(torch.zeros(1, 5, dtype=torch.long), torch.tensor([5]))
    m.train()
    with pytest.raises(v.V100Error):
        m(torch.zeros(1, 50, 64))


def test_state_dict_layout_matches_reference_keys():
    for model, sd in ((v.AudioToTextCTC(64, 128, 29, 128), synth.asr_state_dict(64, 128, 29, 128)),
                      (v.TextToAlignTextModel(29, 64), synth.align_state_dict(29, 64)),
                      (v.AlignTextToAudioModel(29, 64), synth.audio_state_dict(29, 64))):
        assert set(model.state_dict().keys()) == set(sd.keys())
        for k, t in model.state_dict().items():
            assert tuple(t.shape) == tuple(sd[k].shape), k
        model.load_state_dict({k: torch.from_numpy(np.asarray(x)) for k, x in sd.items()})


def test_v2_state_dict_layout_matches_reference_keys():
    small = [list(r) for r in synth.ASR_V2_SMALL_ENCODER]
    dec = [list(r) for r in synth.TTS_V2_BASE_DECODER]
    for model, sd in ((v.AudioToAlignText(64, small, 2, 256, 29), synth.asr_v2_state_dict(64, small, 2, 256, 29)),
                      (v.TextToAlignText(29, 2, 64, 2), synth.align_v2_state_dict(29, 2, 64, 2)),
                      (v.AlignTextToAudio(29, 257, 1, 2, 64, dec), synth.audio_v2_state_dict(29, 257, 1, 2, 64, dec))):
        assert set(model.state_dict().keys()) == set(sd.keys())
        for k, t in model.state_dict().items():
            assert tuple(t.shape) == tuple(sd[k].shape), k
        model.load_state_dict({k: torch.from_numpy(np.asarray(x)) for k, x in sd.items()})


def test_align_v2_host_function_matches_oracle():
    import v100_oracle as orc
    text = torch.from_numpy(synth.text_tokens(3, 17, seed=5))
    align = synth.synthetic_alignment(3, 17, seed=5)
    for i in range(3):
        got = v.TextToAlignText.align(text[i], torch.from_numpy(align[i]))
        assert got.tolist() == orc.align_text_v2(text[i].tolist(), align[i]).tolist()


def test_align_batch_v2_matches_reference_loop():
    import v100_oracle as orc
    text = torch.from_numpy(synth.text_tokens(9, 40, seed=6))
    align = torch.from_numpy(synth.synthetic_alignment(9, 40, seed=6))
    align[3, 5:9, 1] = 0.0                                  # zero durations: the one-frame minimum kicks in
    lens = torch.tensor([40, 1, 17, 40, 33, 2, 40, 25, 9])
    at, at_len = v.align_batch_v2(text, align, lens)
    for b in range(9):
        n = int(lens[b])
        ref = orc.align_text_v2(text[b, :n].tolist(), align[b, :n].numpy())
        assert int(at_len[b]) == len(ref) and at[b, :len(ref)].tolist() == ref.tolist()
        assert (at[b, len(ref):] == 0).all()


def test_align_host_function_matches_oracle():
    import v100_oracle as orc
    text = torch.from_numpy(synth.text_tokens(3, 17, seed=5))
    align = synth.synthetic_alignment(3, 17, seed=5)
    m = v.TextToAlignTextModel(29, 64)
    for i in range(3):
        got = m.align(text[i], torch.from_numpy(align[i]))
        assert got.tolist() == orc.align_text(text[i].tolist(), align[i]).tolist()


def test_align_batch_matches_reference_loop():
    import v100_oracle as orc
    text = torch.from_numpy(synth.text_tokens(9, 40, seed=6))
    align = torch.from_numpy(synth.synthetic_alignment(9, 40, seed=6))
    lens = torch.tensor([40, 1, 17, 40, 33, 2, 40, 25, 9])
    at, at_len = v.align_batch(text, align, lens)
    for b in range(9):
        n = int(lens[b])
        ref = orc.align_text(text[b, :n].tolist(), align[b, :n].numpy())
        assert int(at_len[b]) == len(ref) and at[b, :len(ref)].tolist() == ref.tolist()
        assert (at[b, len(ref):] == 0).all()


def test_sparse_filterbank_roundtrip():
    from voice100_b200.data_modules import mel_filterbank, sparse_filterbank
    fb = mel_filterbank(16000, 512, 64)
    start, count, off, w = sparse_filterbank(fb)
    dense = np.zeros_like(fb)
    for m in range(64):
        dense[start[m]:start[m] + count[m], m] = w[off[m]:off[m] + count[m]]
    assert np.array_equal(dense, fb) and len(w) <= 520 and count.max() <= 24


def test_bench_work_model_matches_survey():
    import sys
    sys.path.insert(0, ROOT)
    import bench
    work = bench.asr_work_model(1, 101, 512, 512, 29, fused=False)   # ~ one audio-second (100 in-frames -> ~50 out)
    gemm = sum(w["flops"] for w in work if w["kind"] == "gemm") / 1e6
    dw = sum(w["flops"] for w in work if w["kind"] == "dwconv") / 1e6
    assert abs(gemm - 1084.6 - 1.48) / 1086 < 0.03 and abs(dw - 72.0) / 72.0 < 0.03, (gemm, dw)
    assert len(work) == 30                                            # log-mel + 9 x 3 + head + CTC tail
    # the fused form (opt-in) charges the same FLOPs, minus the hidden tensor's round trip through HBM
    fused = bench.asr_work_model(1, 101, 512, 512, 29, fused=True)
    assert len(fused) == 22 and abs(sum(w["flops"] for w in fused) - sum(w["flops"] for w in work)) < 1.0
    big = [sum(w["bytes"] for w in bench.asr_work_model(256, 1501, 512, 512, 29, fused=f)) for f in (False, True)]
    assert 22e9 < big[0] < 25e9 and big[1] < 0.65 * big[0]           # ~23.5 GB per 256 x 15 s step, ~14 GB fused


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: integers exactly as float64, floats as float32, and above the size limit the same
    seeded utterances from every array, the same ones on every call."""
    import sys
    sys.path.insert(0, ROOT)
    import bench
    tok = torch.arange(40 * 7, dtype=torch.int64).view(40, 7)
    logits = torch.randn(40, 7, 5, dtype=torch.float16)
    bench.dump_outputs(str(tmp_path / "all"), {"tokens": tok, "logits": logits})
    assert np.load(tmp_path / "all" / "tokens.npy").dtype == np.float64
    assert np.array_equal(np.load(tmp_path / "all" / "tokens.npy"), tok.numpy())
    assert np.array_equal(np.load(tmp_path / "all" / "logits.npy"), logits.float().numpy())
    assert not (tmp_path / "all" / "sample_rows.npy").exists()
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4096)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"tokens": tok, "logits": logits})
        assert sum(f.stat().st_size - 128 for f in (tmp_path / d).iterdir()) <= 4096   # minus the .npy headers
    rows = np.load(tmp_path / "a" / "sample_rows.npy").astype(np.int64)
    assert 0 < len(rows) < 40 and np.array_equal(rows, np.load(tmp_path / "b" / "sample_rows.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "tokens.npy"), tok.numpy()[rows])
    assert np.array_equal(np.load(tmp_path / "b" / "logits.npy"), logits.float().numpy()[rows])


def test_load_checkpoint_roundtrip(tmp_path):
    """Lightning-style .ckpt (state_dict + hyper_parameters, plus training-only keys) -> drop-in module."""
    from collections import OrderedDict
    sd = OrderedDict((k, torch.from_numpy(np.asarray(x))) for k, x in synth.asr_state_dict(64, 128, 44, 128, seed=8).items())
    sd["criterion.dummy"] = torch.zeros(1)      # training-only sub-module state is ignored
    path = tmp_path / "asr.ckpt"
    torch.save({"state_dict": sd, "hyper_parameters": {"audio_size": 64, "embed_size": 128.0, "vocab_size": 44,
                                                       "hidden_size": 128.0, "learning_rate": 1e-3}}, path)
    m = v.load_checkpoint(str(path), device="cpu")
    assert isinstance(m, v.AudioToTextCTC) and not m.training
    assert m.decoder.layers[1].weight.shape == (44, 128, 1)
    assert torch.equal(m.state_dict()["encoder.layers.3.conv.1.0.weight"], sd["encoder.layers.3.conv.1.0.weight"])
    # bare state_dict of the audio model, class inferred from the keys, WORLD statistics from a side file
    au = {k: torch.from_numpy(np.asarray(x)) for k, x in synth.audio_state_dict(29, 64, seed=8).items()}
    stat = {k[len("norm."):]: torch.from_numpy(np.asarray(x)) for k, x in
            synth.audio_state_dict(29, 64, seed=9, randomize_norm=True).items() if k.startswith("norm.")}
    torch.save(au, tmp_path / "audio.pt")
    torch.save(stat, tmp_path / "stat.pt")
    m2 = v.load_checkpoint(str(tmp_path / "audio.pt"), audio_stat=str(tmp_path / "stat.pt"), device="cpu",
                           storage_dtype=torch.float16)
    assert isinstance(m2, v.AlignTextToAudioModel) and m2.storage_dtype == torch.float16
    assert torch.equal(m2.norm.logspc_mean, stat["logspc_mean"])
    with pytest.raises(v.V100Error):
        v.load_checkpoint(str(path), model_class="TextToAlignTextModel", device="cpu")


def test_load_checkpoint_v2(tmp_path):
    """v2 checkpoints (what the reference's shipped configs produce): class from the keys, conv settings from the
    Lightning hyper_parameters (or `hparams=` for a bare state_dict), everything else from the tensors."""
    small = [list(r) for r in synth.ASR_V2_SMALL_ENCODER]
    sd = {k: torch.from_numpy(np.asarray(x)) for k, x in synth.asr_v2_state_dict(64, small, 2, 256, 44, seed=3).items()}
    sd["criterion.dummy"] = torch.zeros(1)
    torch.save({"state_dict": sd, "hyper_parameters": {"audio_size": 64, "encoder_settings": small,
                                                       "decoder_num_layers": 2, "decoder_hidden_size": 256,
                                                       "vocab_size": 44}}, tmp_path / "asr_v2.ckpt")
    m = v.load_checkpoint(str(tmp_path / "asr_v2.ckpt"), device="cpu")
    assert isinstance(m, v.AudioToAlignText) and m.dense.weight.shape == (44, 512) and m.lstm.num_layers == 2
    assert m.encoder[0].conv.stride == (2,) and torch.equal(m.lstm.weight_hh_l1_reverse, sd["lstm.weight_hh_l1_reverse"])
    bare = {k: t for k, t in sd.items() if not k.startswith("criterion")}
    torch.save(bare, tmp_path / "asr_v2_bare.pt")
    with pytest.raises(v.V100Error, match="hparams"):
        v.load_checkpoint(str(tmp_path / "asr_v2_bare.pt"), device="cpu")
    assert isinstance(v.load_checkpoint(str(tmp_path / "asr_v2_bare.pt"), device="cpu",
                                        hparams={"encoder_settings": small}), v.AudioToAlignText)
    wrong = [[256, False, 5, 2, 2, False], [256, False, 3, 1, 1, False]]
    with pytest.raises(v.V100Error, match="disagrees"):
        v.load_checkpoint(str(tmp_path / "asr_v2_bare.pt"), device="cpu", hparams={"encoder_settings": wrong})
    al = {k: torch.from_numpy(np.asarray(x)) for k, x in synth.align_v2_state_dict(29, 2, 64, 2, seed=3).items()}
    torch.save(al, tmp_path / "align_v2.pt")
    m2 = v.load_checkpoint(str(tmp_path / "align_v2.pt"), device="cpu")
    assert isinstance(m2, v.TextToAlignText) and m2.embedding.weight.shape == (29, 64)
    dec = [list(r) for r in synth.TTS_V2_BASE_DECODER]
    au = {k: torch.from_numpy(np.asarray(x)) for k, x in
          synth.audio_v2_state_dict(29, 257, 1, 2, 64, dec, seed=3, randomize_norm=True).items()}
    torch.save({"state_dict": au, "hyper_parameters": {"decoder_settings": dec}}, tmp_path / "tts_v2.ckpt")
    m3 = v.load_checkpoint(str(tmp_path / "tts_v2.ckpt"), device="cpu")
    assert isinstance(m3, v.AlignTextToAudio) and m3.logspc_size == 257 and m3.codeap_size == 1
    assert torch.equal(m3.norm.logspc_mean, au["norm.logspc_mean"])
