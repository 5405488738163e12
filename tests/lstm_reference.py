"""Teacher-forced, error-bounded reference for one bidirectional LSTM layer as `lstm_pair_kernel` computes it.

The kernel's output y[d][t] IS its hidden state h_t rounded to the storage type, and the MMA of the next step consumes
exactly those values.  So instead of running a free reference next to the kernel (whose error then mixes with the
recurrence's own chaotic drift and grows with T), the check feeds every step the kernel's own h_{t-1}:

  * every step's pre-activations at once, a = gx + h_prev @ W_hh^T, in float64 from the exact 16-bit values of gx,
    W_hh and y (one matmul per direction and block of steps);
  * only the cell-state recursion runs step by step, in float64, under the packed-sequence mask t < len[b] (state and
    output are zero outside it, so the reverse direction starts at each utterance's own last step);
  * next to it an element-wise bound B_h[d, t, b, u] on |y - h_ref| that follows the kernel's arithmetic:
      - accumulation: 2 H 2^-24 (|W_hh| |h_prev|) covers an fp32 tensor-core sum of H exact products in any order,
        truncating or not, plus 2^-24 |a| for the fp32 add of the input projection;
      - gates: tanh.approx.f32 has a maximum relative error of about 2^-11 (PTX ISA); the budget is 2^-10 absolute for
        tanh and 2^-11 for sigmoid(x) = tanh(x / 2) / 2 + 1 / 2, plus the pre-activation bound times the slope
        (1 for tanh, 1/4 for sigmoid);
      - cell: c = f c + i g gives  Bc_t = (f + E_f) Bc_{t-1} + |c_{t-1}| E_f + |g| E_i + (i + E_i) E_g  plus the two
        fp32 roundings, then h = o tanh(c) gives  (o + E_o)(min(Bc, 2) + E_tanh) + |tanh c| E_o;
      - output: rounding to the storage type, 2^-8 |y| for bf16 and 2^-11 |y| for fp16 (round to nearest: the error
        is at most the unit roundoff times the ROUNDED value), plus half the smallest fp16 subnormal.
    The bound does not grow with T because h is teacher-forced (only the cell state carries error forward, damped by
    the forget gate), so a single wrong (step, utterance, unit) breaks it by orders of magnitude and is reported by
    its coordinates.
  * exact zeros wherever the output must be zero: t >= len[b], and the padding utterances b in [B, Bp).

Layouts are the kernel's (time-major, csrc/seq.cu): gx [8H, T*Bp] (row d*4H + gate*H + unit, gates i, f, g, o),
w_hh [2, 4H, H], y [2H, T*Bp] (row d*H + unit), column t*Bp + b.  Everything runs on the device of `y`.
"""
from dataclasses import dataclass, field

import torch

E_TANH = 2.0 ** -10              # tanh.approx.f32: max relative error ~2^-11 (PTX ISA), budgeted twice over, absolute
E_SIGMOID = 2.0 ** -11           # sigmoid(x) = tanh.approx(x / 2) / 2 + 1 / 2: half the tanh error
U32 = 2.0 ** -24                 # fp32 unit roundoff
UNIT_ROUNDOFF = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
ABS_FLOOR = {torch.bfloat16: 0.0, torch.float16: 2.0 ** -25}   # fp16 subnormal spacing 2^-24, rounded to nearest
QUANTILE_SAMPLE = 1 << 22        # quantiles of the bound over at most this many (evenly strided) live elements


@dataclass
class LstmCheck:
    """What `check_layer` found.  `ok` = no bound violation, no nonzero where zero is due."""
    violations: int = 0          # live elements with |y - h_ref| > B_h (or a non-finite y)
    nonzero_dead: int = 0        # t >= len[b], b < B, where y != 0 (NaN counts)
    nonzero_pad: int = 0         # b in [B, Bp) where y != 0
    n_live: int = 0
    worst_ratio: float = 0.0     # max |y - h_ref| / B_h over live elements
    worst_at: tuple = ()         # (direction, t, b, unit) of worst_ratio
    first_bad: list = field(default_factory=list)   # up to 5 (direction, t, b, unit, y, h_ref, bound)
    first_step: dict = field(default_factory=dict)  # direction -> its first violated step in processing order
    bound_median: float = 0.0
    bound_p99: float = 0.0
    bound_mean: float = 0.0

    @property
    def ok(self):
        return self.violations == 0 and self.nonzero_dead == 0 and self.nonzero_pad == 0

    def summary(self):
        return (f"worst err/bound {self.worst_ratio:.3f} at (dir, t, b, unit) {self.worst_at}; bound median "
                f"{self.bound_median:.2e} p99 {self.bound_p99:.2e}; {self.violations} violations "
                f"(first step per direction {self.first_step}), "
                f"{self.nonzero_dead} nonzero past the length, {self.nonzero_pad} nonzero padding of {self.n_live} live")

    def assert_ok(self, what=""):
        assert self.ok, f"{what}: {self.summary()}; first violations (dir, t, b, unit, y, ref, bound): {self.first_bad}"


def live_mask(lengths, B, Bp, T, device):
    """[T, Bp] bool: t < len[b] for b < B, False for the padding utterances."""
    ln = torch.zeros(Bp, dtype=torch.long, device=device)
    ln[:B] = torch.as_tensor(lengths, device=device).long()
    return torch.arange(T, device=device)[:, None] < ln[None, :]


def check_layer(y, gx, w_hh, lengths, B, Bp, T, H, dtype, t_chunk=128) -> LstmCheck:
    """Check the layer output `y` [2H, T*Bp] against the teacher-forced float64 recursion; see the module docstring."""
    dev = y.device
    u_out, floor = UNIT_ROUNDOFF[dtype], ABS_FLOOR[dtype]
    live = live_mask(lengths, B, Bp, T, dev)
    is_pad = torch.zeros(Bp, dtype=torch.bool, device=dev)
    is_pad[B:] = True
    r = LstmCheck()
    bounds = []
    worst = (-1.0, ())
    for d in range(2):
        Y = y[d * H:(d + 1) * H].view(H, T, Bp).permute(1, 2, 0).double()              # [T, Bp, H]
        nz = Y != 0
        r.nonzero_pad += int((nz & is_pad[None, :, None]).sum())
        r.nonzero_dead += int((nz & ~live[:, :, None] & ~is_pad[None, :, None]).sum())
        Yl = torch.where(live[:, :, None], Y, 0.0)                                        # what the recursion consumes
        W = w_hh[d].double()                                                              # [4H, H]
        Wa = W.abs()
        G = gx[d * 4 * H:(d + 1) * 4 * H].view(4 * H, T, Bp)
        ref = torch.zeros_like(Y)
        bnd = torch.zeros_like(Y)
        c = torch.zeros(Bp, H, dtype=torch.float64, device=dev)
        Bc = torch.zeros_like(c)
        order = list(range(T)) if d == 0 else list(range(T - 1, -1, -1))
        for k0 in range(0, T, t_chunk):
            steps = order[k0:k0 + t_chunk]
            ts = torch.tensor(steps, device=dev)
            prev = ts - 1 if d == 0 else ts + 1                                           # the step h_prev comes from
            valid = (prev >= 0) & (prev < T)
            hp = Yl[prev.clamp(0, T - 1)] * valid[:, None, None]                          # [n, Bp, H]
            a = G[:, ts].permute(1, 2, 0).double() + hp @ W.T                             # [n, Bp, 4H]
            Ba = 2 * H * U32 * (hp.abs() @ Wa.T) + U32 * a.abs()
            ai, af, ag, ao = a.split(H, dim=-1)
            bi, bf, bg, bo = Ba.split(H, dim=-1)
            gi, gf, gg, go = torch.sigmoid(ai), torch.sigmoid(af), torch.tanh(ag), torch.sigmoid(ao)
            Ei, Ef, Eg, Eo = E_SIGMOID + bi / 4, E_SIGMOID + bf / 4, E_TANH + bg, E_SIGMOID + bo / 4
            for j, t in enumerate(steps):
                lv = live[t][:, None]
                i, f, g, o = gi[j], gf[j], gg[j], go[j]
                cn = f * c + i * g
                Bn = ((f + Ef[j]) * Bc + c.abs() * Ef[j] + g.abs() * Ei[j] + (i + Ei[j]) * Eg[j]
                      + 2 * U32 * ((f + Ef[j]) * (c.abs() + Bc) + (i + Ei[j]) * (g.abs() + Eg[j])))
                th = torch.tanh(cn)
                Bh = (o + Eo[j]) * (Bn.clamp(max=2.0) + E_TANH) + th.abs() * Eo[j] + 2 * U32
                c = torch.where(lv, cn, 0.0)
                Bc = torch.where(lv, Bn, 0.0)
                ref[t] = torch.where(lv, o * th, 0.0)
                bnd[t] = torch.where(lv, Bh, 0.0)
        bnd += u_out * Y.abs() + floor
        err = (Y - ref).abs()
        lv3 = live[:, :, None].expand_as(Y)
        bad = lv3 & ~(err <= bnd)                                                         # NaN / inf is a violation
        r.violations += int(bad.sum())
        bad_t = bad.flatten(1).any(1).nonzero().flatten()
        if bad_t.numel():
            r.first_step[d] = int(bad_t.min()) if d == 0 else int(bad_t.max())
        if len(r.first_bad) < 5 and bool(bad.any()):
            for t, b, u in bad.nonzero()[: 5 - len(r.first_bad)].tolist():
                r.first_bad.append((d, t, b, u, float(Y[t, b, u]), float(ref[t, b, u]), float(bnd[t, b, u])))
        ratio = torch.where(lv3, err / bnd, 0.0).nan_to_num(nan=float("inf"))
        m = float(ratio.max()) if ratio.numel() else 0.0
        if m > worst[0]:
            t, b, u = (int(v) for v in torch.unravel_index(ratio.argmax(), ratio.shape))
            worst = (m, (d, t, b, u))
        bounds.append(bnd[lv3].float())
        r.n_live += int(lv3.sum())
        del Y, Yl, ref, bnd, err, ratio, bad
    r.worst_ratio, r.worst_at = max(worst[0], 0.0), worst[1]
    allb = torch.cat(bounds)
    if allb.numel():
        r.bound_mean = float(allb.double().mean())
        if allb.numel() > QUANTILE_SAMPLE:
            allb = allb[:: (allb.numel() + QUANTILE_SAMPLE - 1) // QUANTILE_SAMPLE]
        q = torch.quantile(allb, torch.tensor([0.5, 0.99], device=allb.device))
        r.bound_median, r.bound_p99 = float(q[0]), float(q[1])
    return r
