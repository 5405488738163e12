"""The teacher-forced LSTM checker (tests/lstm_reference.py) proven on the CPU before it judges the kernel.

A float32 emulation of `lstm_pair_kernel`'s arithmetic (input projection and every h_t rounded to the storage type,
every tanh perturbed by up to the tanh.approx error, 2^-11 relative) must pass the checker at ragged lengths including
0 and T and at batch sizes that are not multiples of 8 or 64; each of the protocol bugs a persistent recurrent kernel
can have must fail it; and the bound must be tight enough (99th percentile below 0.01) to mean something.
"""
import numpy as np
import pytest
import torch

from lstm_reference import check_layer
from voice100_b200 import synth

TANH_APPROX_REL = 2.0 ** -11


def _case(B, T, I, H, dtype, seed):
    """Weights as the v2 models' synthetic checkpoints (gain 2), random inputs, ragged lengths with a 0 and a T.
    -> dict with gx [8H, T*Bp] and w_hh [2, 4H, H] in the storage type, lengths, shapes."""
    Bp = (B + 7) // 8 * 8
    sd = {}
    synth._lstm(sd, seed, "lstm", I, H, 1, 2.0)
    sd = {k: torch.from_numpy(v) for k, v in sd.items()}
    w_ih = torch.cat([sd["lstm.weight_ih_l0"], sd["lstm.weight_ih_l0_reverse"]], 0).to(dtype)
    w_hh = torch.stack([sd["lstm.weight_hh_l0"], sd["lstm.weight_hh_l0_reverse"]], 0).to(dtype)
    bias = (torch.cat([sd["lstm.bias_ih_l0"], sd["lstm.bias_ih_l0_reverse"]], 0) +
            torch.cat([sd["lstm.bias_hh_l0"], sd["lstm.bias_hh_l0_reverse"]], 0)).float()
    g = np.random.Generator(np.random.PCG64(seed))
    x = torch.zeros(I, T, Bp)
    x[:, :, :B] = torch.from_numpy(g.standard_normal((I, T, B)).astype(np.float32)).to(dtype).float()
    gx = (w_ih.float() @ x.view(I, T * Bp) + bias[:, None]).to(dtype)                # the GEMM's rounded output
    lengths = [int(n) for n in g.integers(1, T + 1, size=B)]
    lengths[0], lengths[B // 2], lengths[-1] = T, 0, max(1, T // 3)
    return dict(gx=gx, w_hh=w_hh, lengths=lengths, B=B, Bp=Bp, T=T, H=H, dtype=dtype, seed=seed)


def emulate(case, mutation=None):
    """float32 stand-in for the kernel -> y [2H, T*Bp] in the storage type.  `mutation` injects one bug."""
    gx, w_hh, lengths = case["gx"], case["w_hh"], case["lengths"]
    B, Bp, T, H, dtype = (case[k] for k in ("B", "Bp", "T", "H", "dtype"))
    gen = torch.Generator().manual_seed(case["seed"])
    ln = torch.zeros(Bp, dtype=torch.long)
    ln[:B] = torch.tensor(lengths)
    y = torch.zeros(2 * H, T, Bp, dtype=dtype)
    ragged = next(b for b in range(B) if 0 < lengths[b] < T - 2)                      # an utterance that ends early
    live_pair = [b for b in range(B) if lengths[b] == T][:1] + [b for b in range(B) if lengths[b] >= T // 2 + 2][-1:]

    def tanh(z):
        return torch.tanh(z) * (1 + TANH_APPROX_REL * (2 * torch.rand(z.shape, generator=gen) - 1))

    def sigmoid(z):
        return 0.5 * tanh(0.5 * z) + 0.5

    for d in range(2):
        W = w_hh[d].float()
        G = gx[d * 4 * H:(d + 1) * 4 * H].view(4 * H, T, Bp).float()
        h = torch.zeros(Bp, H)
        c = torch.zeros(Bp, H)
        hist = [h]
        for k in range(T):
            t = k if d == 0 else T - 1 - k
            hp = h
            if mutation == "stale_h" and d == 0 and k == T // 2:
                hp = hist[-2]                                                             # h_{t-2} instead of h_{t-1}
            if mutation == "swap_utterances" and d == 1 and k == T // 2:
                hp = h.clone()
                hp[live_pair] = h[live_pair[::-1]]
            a = G[:, t].T + hp @ W.T                                                      # [Bp, 4H]
            if mutation == "gate_order" and d == 0:
                a = a.clone()                                                             # i <-> f for units 64..127
                a[:, 64:128], a[:, H + 64:H + 128] = a[:, H + 64:H + 128].clone(), a[:, 64:128].clone()
            i, f = sigmoid(a[:, :H]), sigmoid(a[:, H:2 * H])
            gg, o = tanh(a[:, 2 * H:3 * H]), sigmoid(a[:, 3 * H:])
            cn = f * c + i * gg
            hn = o * tanh(cn)
            live = (t < ln)[:, None]
            state_live = live
            if mutation == "reverse_from_end" and d == 1:
                state_live = live.clone()                                                 # runs from T - 1, stores masked
                state_live[ragged] = True
            c = torch.where(state_live, cn, 0.0)
            if mutation == "cell_not_reset" and d == 1:
                c = cn                                                                    # dead steps keep the cell
            h_state = torch.where(state_live, hn, 0.0).to(dtype).float()
            h = torch.where(live, h_state, 0.0)
            y[d * H:(d + 1) * H, t] = h.T.to(dtype)
            if mutation == "reverse_from_end" and d == 1:
                h = h_state
            hist.append(h)
    if mutation == "padding_column":
        y[3, T // 2, Bp - 1] = 2.0 ** -12
    return y.view(2 * H, T * Bp)


def _check(case, y):
    return check_layer(y, case["gx"], case["w_hh"], case["lengths"], case["B"], case["Bp"], case["T"], case["H"],
                       case["dtype"])


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("B,T,I,H", [(70, 120, 64, 128), (13, 40, 32, 192), (130, 9, 64, 64)])
def test_checker_accepts_the_kernel_arithmetic(dtype, B, T, I, H):
    case = _case(B, T, I, H, dtype, seed=B + T)
    assert case["Bp"] > B and B % 64 != 0
    r = _check(case, emulate(case))
    print(dtype, (B, T, I, H), r.summary())
    r.assert_ok("emulated kernel")
    assert 0 < r.worst_ratio < 1.0


def test_bound_is_sharp_at_scale():
    """A 99th percentile far below the size of any protocol bug's effect (an h of the wrong step or utterance moves a
    hidden unit by ~0.1)."""
    case = _case(64 + 6, 300, 128, 256, torch.bfloat16, seed=7)
    r = _check(case, emulate(case))
    print(r.summary())
    r.assert_ok("emulated kernel")
    assert r.bound_p99 < 0.01 and r.bound_median < 0.005, r.summary()


MUTATIONS = ["stale_h", "swap_utterances", "gate_order", "reverse_from_end", "cell_not_reset", "padding_column"]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("mutation", MUTATIONS)
def test_checker_rejects(mutation, dtype):
    case = _case(70, 120, 64, 128, dtype, seed=11)
    r = _check(case, emulate(case, mutation))
    print(mutation, dtype, r.summary())
    assert not r.ok
    if mutation == "padding_column":
        assert r.nonzero_pad == 1 and r.violations == 0
    else:
        # the output past each length stays zero in every one of these: only the bound can see them, and it sees
        # them by a wide margin, at the step where the bug happened
        assert r.nonzero_dead == 0 and r.nonzero_pad == 0
        assert r.worst_ratio > 10, r.summary()
        if mutation == "stale_h":
            assert r.first_step == {0: 120 // 2}
        if mutation == "swap_utterances":
            assert r.first_step == {1: 120 - 1 - 120 // 2}
        if mutation in ("reverse_from_end", "cell_not_reset"):
            assert set(r.first_step) == {1}
