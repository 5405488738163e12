"""`lstm_pair_kernel` step by step at the shapes the v2 models run, against the teacher-forced float64 reference with a
derived element-wise error bound (tests/lstm_reference.py, proven on the CPU by tests/test_lstm_reference_cpu.py).

Each case calls v100_lstm_layer directly, as K.lstm_layer does (input projection by v100_conv1x1), into buffers the test
owns: the output is filled with a NaN pattern the kernel cannot produce and framed by guard bands, so an element the
kernel skips or a write outside the output shows; the workspace is exactly v100_lstm_workspace_bytes, 1024-byte aligned,
between two guard bands.  Every case asserts error <= bound on every live element, exact zeros past each length and in
the padding utterances, every output element written and untouched guard bands, and prints its worst error/bound ratio
with the bound's median and 99th percentile.  Needs a CUDA device (-m gpu).
"""
import numpy as np
import pytest
import torch

from lstm_reference import check_layer
from voice100_b200 import _lib, synth, v2
from voice100_b200 import kernels as K

pytestmark = pytest.mark.gpu
DEV = "cuda"
BF16, F16 = torch.bfloat16, torch.float16
DTYPES = [BF16, F16]
SENTINEL = {BF16: 0x7FA5, F16: 0x7D5A}    # non-canonical NaNs (hardware NaNs are canonical)
GUARD_BYTES = 4096
GUARD_BYTE = 0xA5


class OwnedOut:
    """[2H, T*Bp] layer output, sentinel-filled, GUARD_BYTES of guard band on both sides."""

    def __init__(self, rows, cols, dtype):
        self.dtype, self.g, self.n = dtype, GUARD_BYTES // 2, rows * cols
        self.raw = torch.empty((self.g + self.n + self.g,), dtype=torch.int16, device=DEV)
        self.t = self.raw[self.g:self.g + self.n].view(dtype).view(rows, cols)
        self.reset()

    def reset(self):
        self.raw.fill_(SENTINEL[self.dtype])

    def ptr(self):
        return self.t.data_ptr()

    def check(self, what):
        s = SENTINEL[self.dtype]
        for side, band in (("before", self.raw[:self.g]), ("after", self.raw[self.g + self.n:])):
            assert int((band != s).sum()) == 0, f"{what}: the guard band {side} the output was written"
        n_skip = int((self.t.view(torch.int16) == s).sum())
        assert n_skip == 0, f"{what}: {n_skip} of {self.n} output elements were never written"


class OwnedWorkspace:
    """Exactly v100_lstm_workspace_bytes(B, H), 1024-byte aligned, between two guard bands."""

    def __init__(self, B, H):
        self.n = int(_lib.lib().v100_lstm_workspace_bytes(B, H))
        self.raw = torch.full((GUARD_BYTES + 1024 + self.n + GUARD_BYTES,), GUARD_BYTE, dtype=torch.uint8, device=DEV)
        self.off = GUARD_BYTES + (-(self.raw.data_ptr() + GUARD_BYTES)) % 1024
        self.ws = self.raw[self.off:self.off + self.n]
        assert self.ws.data_ptr() % 1024 == 0

    def ptr(self):
        return self.ws.data_ptr()

    def check(self, what):
        for side, band in (("before", self.raw[:self.off]), ("after", self.raw[self.off + self.n:])):
            n = int((band != GUARD_BYTE).sum())
            assert n == 0, f"{what}: {n} bytes of the guard band {side} the workspace were written"


def weights(I, H, dtype, seed):
    """One bidirectional layer of a synthetic v2 checkpoint (gain 2), in the layout K.lstm_layer takes."""
    sd = {}
    synth._lstm(sd, seed, "lstm", I, H, 1, 2.0)
    sd = {k: torch.from_numpy(v) for k, v in sd.items()}
    w_ih = torch.cat([sd["lstm.weight_ih_l0"], sd["lstm.weight_ih_l0_reverse"]], 0).to(DEV, dtype).contiguous()
    w_hh = torch.stack([sd["lstm.weight_hh_l0"], sd["lstm.weight_hh_l0_reverse"]], 0).to(DEV, dtype).contiguous()
    bias = (torch.cat([sd["lstm.bias_ih_l0"], sd["lstm.bias_ih_l0_reverse"]], 0) +
            torch.cat([sd["lstm.bias_hh_l0"], sd["lstm.bias_hh_l0_reverse"]], 0)).to(DEV).float().contiguous()
    return dict(w_ih=w_ih, w_hh=w_hh, bias=bias)


def frame_lengths(B, T, seed):
    """The benchmark's clip lengths, U[2 s, 15 s] at 16 kHz, as encoder frames (n // 160 + 2) // 2 (751 for 15 s),
    scaled to T steps; the last utterance has T steps and the second none."""
    n = synth.ragged_lengths(B, 2 * 16000, 15 * 16000, seed=seed).astype(np.int64)
    f = np.minimum((n // 160 + 2) // 2 * T // 751, T)
    f[-1] = T
    if B > 1:
        f[1] = 0
    return [int(v) for v in f]


def tm_input(B, I, T, dtype, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn((B, I, T), generator=g, device=DEV)
    return K.ncw_to_tm(K.ncw_from_f32(x, dtype))


class Layer:
    """One direct v100_lstm_layer call: input projection, owned output and workspace."""

    def __init__(self, x: K.Tm, w, lengths, ws: OwnedWorkspace = None):
        self.x, self.w, self.lengths = x, w, list(lengths)
        self.H = w["w_hh"].shape[2]
        self.dtype = x.data.dtype
        self.len_dev = torch.tensor(self.lengths, dtype=torch.int32, device=DEV)
        self.gx = K.conv1x1(x.as_ncw(), w["w_ih"], None, w["bias"], K.ACT_NONE)      # [1, 8H, T*Bp], as K.lstm_layer
        self.ws = ws if ws is not None else OwnedWorkspace(x.B, self.H)
        self.y = OwnedOut(2 * self.H, x.T * x.Bp, self.dtype)

    def launch(self, y_ptr=None):
        x = self.x
        K._call(x, "v100_lstm_layer", self.gx.data.data_ptr(), self.w["w_hh"].data_ptr(), self.len_dev.data_ptr(),
                self.y.ptr() if y_ptr is None else y_ptr, self.ws.ptr(), x.B, x.Bp, x.T, self.H, K.dt(self.dtype))

    def out(self) -> K.Tm:
        return K.Tm(self.y.t, self.x.B, self.x.T, self.x.Bp)

    def check(self, what):
        torch.cuda.synchronize()
        self.y.check(what)
        self.ws.check(what)
        x = self.x
        r = check_layer(self.y.t, self.gx.data.view(8 * self.H, x.T * x.Bp), self.w["w_hh"], self.lengths, x.B, x.Bp,
                        x.T, self.H, self.dtype)
        print(f"\n{what}: {r.summary()}")
        r.assert_ok(what)
        return r


def _name(dtype):
    return "bf16" if dtype == BF16 else "fp16"


# ------------------------------------------------------------------------------------------------
# the model shapes
# ------------------------------------------------------------------------------------------------
ASR = dict(B=256, T=751, H=512)


@pytest.fixture(scope="module", params=DTYPES, ids=_name)
def asr_layers(request):
    """AudioToAlignText's two layers at the benchmark shape (256 x 15 s): layer 2 is fed layer 1's output."""
    dtype = request.param
    B, T, H = ASR["B"], ASR["T"], ASR["H"]
    lengths = frame_lengths(B, T, seed=1234)
    x = tm_input(B, H, T, dtype, seed=1)
    w1, w2 = weights(H, H, dtype, seed=21), weights(2 * H, H, dtype, seed=22)
    l1 = Layer(x, w1, lengths)
    l1.launch()
    l2 = Layer(l1.out(), w2, lengths)
    l2.launch()
    return dtype, l1, l2


def test_asr_v2_layers(asr_layers):
    dtype, l1, l2 = asr_layers
    l1.check(f"asr_v2 layer 1 {_name(dtype)} B=256 T=751 512->512")
    l2.check(f"asr_v2 layer 2 {_name(dtype)} B=256 T=751 1024->512")


@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_align_v2(dtype):
    """TextToAlignText: H = 256, 100 steps."""
    B, T, H = 256, 100, 256
    layer = Layer(tm_input(B, H, T, dtype, seed=3), weights(H, H, dtype, seed=31), frame_lengths(B, T, seed=5))
    layer.launch()
    layer.check(f"align_v2 {_name(dtype)} B=256 T=100 256->256")


@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_tts_v2_long(dtype):
    """AlignTextToAudio with max_frames: 1000 steps, every utterance shorter than T, some empty; a ragged last group."""
    B, T, H = 200, 1000, 512
    g = np.random.Generator(np.random.PCG64(41))
    lengths = [int(v) for v in g.integers(T // 4, T, size=B)]
    for b in (0, 77, B - 1):
        lengths[b] = 0
    lengths[5] = T - 1
    layer = Layer(tm_input(B, H, T, dtype, seed=4), weights(H, H, dtype, seed=42), lengths)
    layer.launch()
    layer.check(f"tts_v2 long {_name(dtype)} B=200 T=1000 512->512")


@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
def test_multi_launch(dtype):
    """More 64-utterance groups than one cooperative launch holds: the host splits the layer into several launches
    that share the counters and exchange buffers of one workspace."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    H, T = 512, 200
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    g = (sms // 2) // (2 * H // 64)            # groups that fit at one CTA per SM, clusters of two, 16 clusters a group
    B = 64 * (g + 1)
    layer = Layer(tm_input(B, 64, T, dtype, seed=6), weights(64, H, dtype, seed=61), frame_lengths(B, T, seed=7))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        layer.launch()
        torch.cuda.synchronize()
    n = sum(1 for e in prof.events() if e.device_type == DeviceType.CUDA and "lstm_pair_kernel" in e.name)
    print(f"\nmulti-launch: {sms} SMs, B={B} ({g + 1} groups): {n} lstm_pair_kernel launches")
    assert n >= 2, n
    layer.check(f"multi-launch {_name(dtype)} B={B} T=200 64->512")


@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
@pytest.mark.parametrize("H", list(range(64, 513, 64)))
def test_every_hidden_size(H, dtype):
    """Every TMEM column allocation (128 / 256 / 512) and k-block count, one and three groups with a ragged last."""
    for B in (65, 130):
        T = 64
        layer = Layer(tm_input(B, 64, T, dtype, seed=H + B), weights(64, H, dtype, seed=H), frame_lengths(B, T, seed=B))
        layer.launch()
        layer.check(f"H={H} {_name(dtype)} B={B} T=64 64->{H}")


@pytest.mark.parametrize("dtype", DTYPES, ids=_name)
@pytest.mark.parametrize("B,T", [(1, 1), (1, 2), (255, 1), (255, 2)])
def test_edges(B, T, dtype):
    lengths = frame_lengths(B, T, seed=B + T)
    layer = Layer(tm_input(B, 64, T, dtype, seed=B), weights(64, 512, dtype, seed=T), lengths)
    layer.launch()
    layer.check(f"edge {_name(dtype)} B={B} T={T} 64->512")


# ------------------------------------------------------------------------------------------------
# composition, determinism, graph capture, layout
# ------------------------------------------------------------------------------------------------
def test_two_layer_stack_matches_direct_calls(asr_layers):
    """v2._run_lstm (both layers on one shared workspace) = the two direct calls, bit for bit."""
    dtype, l1, l2 = asr_layers
    got = v2._run_lstm(l1.x, [l1.w, l2.w], l1.len_dev)
    torch.cuda.synchronize()
    assert torch.equal(got.data.view(torch.int16), l2.y.t.view(torch.int16))


def test_deterministic_across_launches_and_workspace_reuse():
    """50 launches at the asr_v2 shape, each followed by a different-shaped layer on the same workspace (other group
    count, other H, other T): every output equals the first bit for bit."""
    dtype = BF16
    B, T, H = ASR["B"], ASR["T"], ASR["H"]
    a = Layer(tm_input(B, H, T, dtype, seed=8), weights(H, H, dtype, seed=81), frame_lengths(B, T, seed=9))
    b = Layer(tm_input(130, 64, 64, dtype, seed=10), weights(64, 256, dtype, seed=82), frame_lengths(130, 64, seed=11),
              ws=a.ws)
    a.launch()
    first = a.y.t.view(torch.int16).clone()
    mismatches = torch.zeros((), dtype=torch.int64, device=DEV)
    for _ in range(50):
        b.launch()
        a.y.reset()
        a.launch()
        mismatches += (a.y.t.view(torch.int16) != first).sum()
    torch.cuda.synchronize()
    assert int(mismatches) == 0, f"{int(mismatches)} output elements differ from the first launch over 50 launches"
    a.check("determinism bf16 B=256 T=751 512->512 (last launch)")


def test_graph_capture_replays_the_eager_result():
    dtype = BF16
    B, T, H = 256, 100, 256
    layer = Layer(tm_input(B, H, T, dtype, seed=12), weights(H, H, dtype, seed=121), frame_lengths(B, T, seed=13))
    layer.launch()
    torch.cuda.synchronize()
    eager = layer.y.t.view(torch.int16).clone()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        layer.launch()
    for i in range(3):
        layer.y.reset()
        graph.replay()
        torch.cuda.synchronize()
        layer.y.check(f"graph replay {i}")
        assert torch.equal(layer.y.t.view(torch.int16), eager), f"graph replay {i} differs from the eager call"
    layer.ws.check("graph replay")


def test_layout_round_trip_at_the_model_shape():
    """ncw_to_tm / tm_to_ncw at 256 x 1024 channels x 751 steps: bit exact, NaN in the NCW pitch padding is not read,
    the padding utterances of the time-major tensor are zero and the NCW pitch padding is written as zero."""
    B, C, T = 256, 1024, 751
    g = torch.Generator(device=DEV).manual_seed(14)
    x = K.empty_ncw(B, C, T, DEV, BF16)
    assert x.pitch > T
    x.data.fill_(float("nan"))
    x.data[:, :, :T] = torch.randn((B, C, T), generator=g, device=DEV).to(BF16)
    tm = K.ncw_to_tm(x)
    assert tm.Bp == 256 and tm.data.shape == (C, T * 256)
    assert torch.equal(tm.data.view(C, T, 256).permute(2, 0, 1).view(torch.int16), x.data[:, :, :T].view(torch.int16))
    back = K.tm_to_ncw(tm)
    assert torch.equal(back.data[:, :, :T].view(torch.int16), x.data[:, :, :T].view(torch.int16))
    assert int((back.data[:, :, T:].view(torch.int16) != 0).sum()) == 0
    # a batch that does not fill its last 8: the padding utterances of the time-major tensor are zero
    xs = K.Ncw(x.data[:250].contiguous(), T)
    tms = K.ncw_to_tm(xs)
    v = tms.data.view(C, T, 256)
    assert int((v[:, :, 250:].view(torch.int16) != 0).sum()) == 0
    assert torch.equal(v[:, :, :250].permute(2, 0, 1).view(torch.int16), xs.data[:, :, :T].view(torch.int16))
