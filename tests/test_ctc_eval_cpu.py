"""CPU checks of the ASR evaluation wrappers: argument validation that raises before any launch (the same exception
classes torch.nn.functional.ctc_loss raises), no CPU path, and the reference DPs the GPU tests compare against."""
import numpy as np
import pytest
import torch

import voice100_b200 as v
from ctc_eval_reference import edit_distance_np, edit_distance_py


def _args(T=10, B=3, V=5, S=4):
    return torch.zeros(T, B, V), torch.ones(B, S, dtype=torch.int64), [T] * B, [2] * B


def test_ctc_loss_needs_cuda():
    lp, tg, il, tl = _args()
    with pytest.raises(v.V100Error):
        v.ctc_loss(lp, tg, il, tl)
    with pytest.raises(v.V100Error):
        v.ctc_loss(lp, tg, torch.tensor(il), torch.tensor(tl), reduction="none")


@pytest.mark.parametrize("il,tl,match", [
    ([11, 10, 10], [2, 2, 2], "at most 10"),
    ([-1, 10, 10], [2, 2, 2], "at least 0"),
    ([10, 10, 10], [2, -1, 2], "at least 0"),
    ([10, 10, 10], [2, 5, 2], "size at least 5"),
    ([10, 10], [2, 2, 2], "batch_size"),
])
def test_ctc_loss_host_lengths_raise_like_torch(il, tl, match):
    lp, tg, _, _ = _args()
    for lengths in ((il, tl), (torch.tensor(il), torch.tensor(tl))):
        with pytest.raises(RuntimeError, match=match):
            v.ctc_loss(lp, tg, *lengths)


def test_ctc_loss_concatenated_targets_too_short_raises():
    lp = torch.zeros(10, 3, 5)
    with pytest.raises(RuntimeError, match="size at least 7"):
        v.ctc_loss(lp, torch.ones(6, dtype=torch.int64), [10] * 3, [2, 3, 2])


def test_ctc_loss_blank_and_reduction_checks():
    lp, tg, il, tl = _args()
    with pytest.raises(RuntimeError, match="blank"):
        v.ctc_loss(lp, tg, il, tl, blank=5)
    with pytest.raises(ValueError):
        v.ctc_loss(lp, tg, il, tl, reduction="avg")
    with pytest.raises(v.V100Error):
        v.ctc_loss(lp.double(), tg, il, tl)


def test_edit_distance_needs_cuda():
    x = torch.zeros(2, 4, dtype=torch.int64)
    with pytest.raises(v.V100Error):
        v.edit_distance(x, None, x, None)


def test_reference_dps_agree():
    rng = np.random.default_rng(0)
    cases = [([], []), ([1, 2, 3], []), ([], [4]), ([1, 2, 3], [1, 2, 3]), ([1, 2], [3, 4, 5]),
             (list("kitten"), list("sitting"))]
    for _ in range(200):
        k = int(rng.integers(2, 6))
        cases.append((rng.integers(0, k, int(rng.integers(0, 30))).tolist(),
                      rng.integers(0, k, int(rng.integers(0, 30))).tolist()))
    for a, b in cases:
        ai = [ord(c) if isinstance(c, str) else c for c in a]
        bi = [ord(c) if isinstance(c, str) else c for c in b]
        assert edit_distance_np(ai, bi) == edit_distance_py(ai, bi) == edit_distance_py(bi, ai)
    assert edit_distance_py(list("kitten"), list("sitting")) == 3
