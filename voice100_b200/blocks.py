"""Inverted-residual stacks evaluated with the libv100 kernels.

Parameters live in stock torch containers (nn.Conv1d / nn.BatchNorm1d / nn.ConvTranspose1d /
nn.Embedding instances that are never *called*) so that constructor-time initialisation, `.to()`,
`state_dict()` and `load_state_dict()` behave exactly like the reference's modules and use its key
layout (voice100/models/asr.py:27-59).  `forward` never touches those containers: it runs the folded,
bf16-packed copies built by `prepare_*` through the C ABI.
"""
from __future__ import annotations

from typing import Tuple

import torch
from torch import nn

from . import kernels as K
from ._lib import V100Error

BN_EPS = 1e-5


def fold_bn(bn: nn.BatchNorm1d) -> Tuple[torch.Tensor, torch.Tensor]:
    """Eval-mode BatchNorm1d as y = scale*x + shift, folded in fp32 (asr.py:36,52)."""
    scale = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
    shift = bn.bias.detach().float() - bn.running_mean.detach().float() * scale
    return scale.contiguous(), shift.contiguous()


class InvertedResidualParams(nn.Module):
    """Parameter container with the reference's `conv.{0.0,0.1,1.0,1.1,2,3}` key layout."""

    def __init__(self, c_in: int, c_out: int, kernel_size: int, stride: int = 1, use_residual: bool = True):
        super().__init__()
        h = c_in * 4
        self.c_in, self.c_out, self.hidden = c_in, c_out, h
        self.kernel_size, self.stride, self.use_residual = kernel_size, stride, use_residual
        pad = (kernel_size - 1) // 2
        expand = nn.Sequential(nn.Conv1d(c_in, h, 1, bias=False), nn.BatchNorm1d(h))
        depthwise = nn.Sequential(nn.Conv1d(h, h, kernel_size, stride=stride, padding=pad, groups=h, bias=False),
                                  nn.BatchNorm1d(h))
        self.conv = nn.Sequential(expand, depthwise, nn.Conv1d(h, c_out, 1, bias=False), nn.BatchNorm1d(c_out))

    def forward(self, *a, **k):  # pragma: no cover
        raise V100Error("InvertedResidualParams only stores weights; run the owning model's forward")

    def prepare(self, dtype=torch.bfloat16):
        """-> dict of device tensors the kernels consume (16-bit weights, fp32 folded BN)."""
        e, d, p, bn3 = self.conv[0], self.conv[1], self.conv[2], self.conv[3]
        s1, b1 = fold_bn(e[1])
        s2, b2 = fold_bn(d[1])
        s3, b3 = fold_bn(bn3)
        return dict(
            w1=e[0].weight.detach()[:, :, 0].to(dtype).contiguous(), s1=s1, b1=b1,
            wd=d[0].weight.detach()[:, 0, :].to(dtype).contiguous(), s2=s2, b2=b2,
            w2=p.weight.detach()[:, :, 0].to(dtype).contiguous(), s3=s3, b3=b3,
            k=self.kernel_size, stride=self.stride, res=self.use_residual)


# Read by bench.py's per-kernel work model: expand and depthwise run as two kernels (DESIGN.md section 3.7).
FUSE_EXPAND_DW = False


def run_inverted_residual(x: K.Ncw, w: dict) -> K.Ncw:
    """pw-expand (+BN+ReLU6) -> depthwise k (+BN+ReLU6) -> pw-project (+BN) (+x)   (asr.py:45-59)."""
    h = K.conv1x1(x, w["w1"], w["s1"], w["b1"], K.ACT_RELU6)
    h = K.dwconv(h, w["wd"], w["s2"], w["b2"], w["k"], w["stride"], K.ACT_RELU6)
    return K.conv1x1(h, w["w2"], w["s3"], w["b3"], K.ACT_NONE, res=x if w["res"] else None)


class PreparedCache:
    """Rebuild the packed weights only when a parameter/buffer changed (pointer or in-place version)."""

    def __init__(self, owner: nn.Module, build):
        self._owner, self._build, self._key, self._val = owner, build, None, None

    def get(self):
        key = (getattr(self._owner, "storage_dtype", None),) + tuple(
            (t.data_ptr(), t._version) for t in list(self._owner.parameters()) + list(self._owner.buffers()))
        if key != self._key:
            with torch.no_grad():
                self._val = self._build()
            self._key = key
        return self._val


class StorageDtypeMixin:
    """`storage_dtype` = the 16-bit type activations and weights are stored in: torch.bfloat16 (default, the
    type BASELINE.json's north_star names) or torch.float16 (same tensor-core speed, 8x smaller storage error;
    safe here because every stored activation is bounded by ReLU6 / BatchNorm)."""
    storage_dtype = torch.bfloat16

    def set_storage_dtype(self, dtype):
        K.dt(dtype)
        for m in self.modules():
            if isinstance(m, StorageDtypeMixin):
                m.storage_dtype = dtype
        return self


def require_eval_cuda(module: nn.Module, *tensors: torch.Tensor):
    if module.training:
        raise V100Error(f"{type(module).__name__} is inference-only (BatchNorm uses running statistics): "
                        "call .eval() first")
    for t in tensors:
        if not t.is_cuda:
            raise V100Error(f"{type(module).__name__} runs only on a CUDA device (sm_100a); there is no CPU path")
