"""Resampling on the host side: the tap table is torchaudio's bit for bit, its packing drops only (near-)zero taps,
the restatement oracle/resample.py reproduces torchaudio's outputs, and the output length is torchaudio's.
No GPU needed."""
import math

import numpy as np
import pytest
import torch

import resample as R
from helpers import golden
from voice100_b200 import V100Error
from voice100_b200 import data_modules as dm

RATIOS = [(48000, 16000), (44100, 16000), (32000, 16000), (24000, 16000), (22050, 16000), (11025, 16000),
          (8000, 16000), (16000, 22050), (16000, 24000), (16000, 44100), (16000, 48000)]
METHODS = ("sinc_interp_hann", "sinc_interp_kaiser")
KAISER_DROP_BOUND = 1e-21          # pack_resample_kernel's stated bound for the default beta


def _tag(a, b, lpw=6, rolloff=0.99, method="sinc_interp_hann"):
    return f"{a}_{b}_{lpw}_{rolloff}_{method.split('_')[-1]}"


@pytest.mark.parametrize("rolloff", [0.99, 0.945])
@pytest.mark.parametrize("lpw", [6, 16])
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("a,b", RATIOS)
def test_taps_bit_identical_to_torchaudio(a, b, method, lpw, rolloff):
    F = pytest.importorskip("torchaudio.functional.functional")
    g = math.gcd(a, b)
    ref, width = F._get_sinc_resample_kernel(a, b, g, lpw, rolloff, method, None)
    kernel, w, inside = dm.sinc_resample_kernel(a, b, g, lpw, rolloff, method, None)
    assert w == width and kernel.dtype == torch.float32
    assert torch.equal(kernel.view(torch.int32), ref.view(torch.int32))


@pytest.mark.parametrize("rolloff", [0.99, 0.945])
@pytest.mark.parametrize("lpw", [6, 16])
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("a,b", RATIOS)
def test_packing_drops_only_zero_or_bounded_taps(a, b, method, lpw, rolloff):
    g = math.gcd(a, b)
    kernel, w, inside = dm.sinc_resample_kernel(a, b, g, lpw, rolloff, method, None)
    start, count, off, taps = dm.pack_resample_kernel(kernel, inside)
    k = kernel[:, 0].numpy()
    n, K = k.shape
    assert n == b // g and K == 2 * w + a // g
    assert off[0] == 0 and (off[1:] == off[:-1] + count[:-1]).all() and off[-1] + count[-1] == len(taps)
    for p in range(n):
        s, c = int(start[p]), int(count[p])
        assert c > 0 and s >= 0 and s + c <= K
        assert inside[p].nonzero().flatten().tolist() == list(range(s, s + c))      # one contiguous run
        assert np.array_equal(taps[off[p]:off[p] + c].view(np.int32), k[p, s:s + c].view(np.int32))
        dropped = np.concatenate([k[p, :s], k[p, s + c:]])
        if method == "sinc_interp_hann":
            assert (dropped == 0).all() and (k[p, s:s + c] != 0).all()               # exactly the non-zero taps
        else:
            assert np.abs(dropped).max(initial=0) <= KAISER_DROP_BOUND


def test_tables_equal_the_golden():
    gd = golden("resample")
    tags = sorted({k.split("/")[1] for k in gd.files if k.startswith("table/")})
    assert len(tags) == 24
    for t in tags:
        a, b, lpw, ro, m = t.split("_")
        a, b, lpw, ro = int(a), int(b), int(lpw), float(ro)
        g = math.gcd(a, b)
        kernel, w, inside = dm.sinc_resample_kernel(a, b, g, lpw, ro, "sinc_interp_" + m)
        assert w == int(gd[f"table/{t}/width"])
        for name, arr in zip(("start", "count", "off", "taps"), dm.pack_resample_kernel(kernel, inside)):
            assert np.array_equal(arr, gd[f"table/{t}/{name}"]), (t, name)


def test_restatement_matches_torchaudio_golden():
    """The float64 restatement over the packed fp32 taps against torchaudio's fp32 conv1d: torchaudio's own rounding
    is what remains (up to 1.2e-5 of max|y| at 22.05 kHz)."""
    gd = golden("resample")
    keys = [k for k in gd.files if k.startswith("y/")]
    assert len(keys) == 24
    for key in keys:
        _, ab, L = key.split("/")
        a, b = map(int, ab.split("_"))
        g, t = math.gcd(a, b), _tag(a, b)
        x = gd[f"x/{ab}/{L}"][None]
        y, ol = R.resample_packed(x, [x.shape[1]], gd[f"table/{t}/start"], gd[f"table/{t}/count"], gd[f"table/{t}/off"],
                                  gd[f"table/{t}/taps"], a // g, b // g, int(gd[f"table/{t}/width"]))
        ref = gd[key].astype(np.float64)
        assert y.shape == (1, len(ref)) and ol.tolist() == [len(ref)]
        assert np.abs(y[0] - ref).max() <= 2e-5 * np.abs(ref).max(), key


def test_restatement_zero_pads_past_each_length():
    tab = dm.pack_resample_kernel(*dm.sinc_resample_kernel(44100, 16000, 100)[::2])
    x = np.random.default_rng(1).standard_normal((3, 900)).astype(np.float32)
    x2 = x.copy()
    x2[1, 500:] = 1e30                                       # padding content must not reach a result
    y1, l1 = R.resample_packed(x, [900, 500, 0], *tab, 441, 160, 19 * 441 // 160 + 1)
    y2, l2 = R.resample_packed(x2, [900, 500, 0], *tab, 441, 160, 19 * 441 // 160 + 1)
    assert l1.tolist() == [327, 182, 0] and np.array_equal(y1, y2) and (y1[1, 182:] == 0).all() and (y1[2] == 0).all()
    one, _ = R.resample_packed(x[1:2, :500], [500], *tab, 441, 160, 19 * 441 // 160 + 1)
    assert np.array_equal(one[0], y1[1, :182])


@pytest.mark.parametrize("a,b", RATIOS + [(44100, 8000), (3, 7)])
def test_out_length_is_torchaudio_float_ceil(a, b):
    """resampled_length equals torchaudio's output length, min(torch.ceil(torch.as_tensor(new * length / orig)),
    new * (length // orig + 1)) with reduced rates, for divisible and non-divisible lengths up to 2^31 - 1.
    torch.as_tensor makes the quotient a float32 tensor, so this is not always the exact ceil(n L / o)."""
    g = math.gcd(a, b)
    o, n = a // g, b // g
    rng = np.random.default_rng(a * 7 + b)
    top = 2 ** 31 - 1
    lengths = set(int(v) for v in rng.integers(0, top, 400))
    lengths |= {0, 1, 2, o - 1, o, o + 1, top, top - 1, top - o}
    lengths |= {int(v) * o for v in rng.integers(0, top // o, 200)}             # divisible: n L / o is an integer
    lengths |= {int(v) * o + d for v in rng.integers(1, top // o - 1, 100) for d in (-1, 1)}
    lengths = sorted(v for v in lengths if 0 <= v <= top)
    exact_differs = 0
    for L in lengths:
        ref = min(int(torch.ceil(torch.as_tensor(n * L / o)).long()), n * (L // o + 1))
        assert dm.resampled_length(L, a, b) == ref == R.out_length(L, o, n), L
        exact = (n * L + o - 1) // o
        exact_differs += ref != exact
        assert abs(ref - exact) <= 1 + n * L / o * 2 ** -24, L            # float32 rounding of the quotient
        if n * L / o < 2 ** 22 / o:                          # float32 resolves 1/o here: the exact ceiling
            assert ref == exact, L
    if o > 1:
        assert exact_differs > 0                             # the float32 rounding is real within int32 lengths
    t = torch.tensor(lengths, dtype=torch.int64)
    assert dm.resampled_length(t, a, b).tolist() == [dm.resampled_length(L, a, b) for L in lengths]


def test_argument_errors_match_torchaudio():
    x = torch.zeros(10)
    with pytest.raises(ValueError):
        dm.resample(x, 0, 16000)
    with pytest.raises(ValueError):
        dm.resample(x, 16000, -1)
    with pytest.raises(Exception, match="integer"):
        dm.resample_table(44100.5, 16000, device="cpu")
    with pytest.raises(ValueError, match="Low pass filter width"):
        dm.resample_table(44100, 16000, lowpass_filter_width=0, device="cpu")
    with pytest.raises(ValueError, match="Invalid resampling method"):
        dm.resample_table(44100, 16000, resampling_method="linear", device="cpu")
    with pytest.raises(V100Error):                         # a CPU tensor: there is no host path
        dm.resample(x, 44100, 16000)
    with pytest.raises(V100Error):
        dm.resample(x, 16000, 16000)
