"""compressai.layers / compressai.ops / compressai.models.utils surface on top of the CUDA kernels.

Same constructor signatures, attribute names and state_dict layout as the reference
(compressai/layers/gdn.py, layers/layers.py, ops/bound_ops.py, ops/parametrizers.py,
models/utils.py:128-146), so `coremasic/mywork/MASIC.py` builds its model out of these
classes unchanged.  The parameter containers subclass nn.Conv2d / nn.ConvTranspose2d to
draw the same random init in the same order; their forward() runs the sm_100a kernels on
NCHW fp32 CUDA tensors (inference).  CPU tensors raise: there is no fallback path.
"""
from __future__ import annotations

from typing import Any, Dict, Optional, Tuple

import torch
import torch.nn as nn
from torch import Tensor

from . import _lib, ops
from ._lib import MasicError
from .convplan import (ACT_NONE, CONV, DECONV_S2, DECONV_S2_SUBPIX, GDN_FWD, GDN_INV, GDN_NONE, MASK_A_5x5,
                       ConvPlan, PackedConv)

F16 = _lib.FMT_F16              # inference runs on fp16 operands / activations (csrc/cvt16.cuh)
ACT = _lib.act_dtype(F16)

__all__ = ["GDN", "MaskedConv2d", "ResidualBlock", "conv3x3", "conv1x1", "LowerBound",
           "NonNegativeParametrizer", "conv", "deconv"]


def _require_inference(mod: nn.Module, x: Tensor) -> None:
    if not x.is_cuda:
        raise MasicError(f"{type(mod).__name__}: masic_b200 kernels need CUDA tensors (no CPU fallback)")
    if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in mod.parameters())) \
            and mod.training:
        raise MasicError(f"{type(mod).__name__}: the sm_100a path implements inference (eval / no_grad); "
                         "backward kernels are not built yet (DESIGN.md, section 'out of scope')")


# ----------------------------------------------------------------------------- ops
class LowerBound(nn.Module):
    """compressai/ops/bound_ops.py:60-80 — max(x, bound); forward only on this path."""
    bound: Tensor

    def __init__(self, bound: float):
        super().__init__()
        self.register_buffer("bound", torch.Tensor([float(bound)]))

    def forward(self, x):
        return torch.max(x, self.bound)


class NonNegativeParametrizer(nn.Module):
    """compressai/ops/parametrizers.py:38-64."""
    pedestal: Tensor

    def __init__(self, minimum: float = 0, reparam_offset: float = 2 ** -18):
        super().__init__()
        self.minimum = float(minimum)
        self.reparam_offset = float(reparam_offset)
        pedestal = self.reparam_offset ** 2
        self.register_buffer("pedestal", torch.Tensor([pedestal]))
        bound = (self.minimum + self.reparam_offset ** 2) ** 0.5
        self.lower_bound = LowerBound(bound)

    def init(self, x: Tensor) -> Tensor:
        return torch.sqrt(torch.max(x + self.pedestal, self.pedestal))

    def forward(self, x: Tensor) -> Tensor:
        out = self.lower_bound(x)
        return out ** 2 - self.pedestal


# ----------------------------------------------------------------------------- conv modules
def _to_nhwc_bf16(x: Tensor, pitch: int) -> Tensor:
    """NCHW fp32 -> NHWC bf16 with `pitch` channels (layout plumbing between unfused modules)."""
    n, c, h, w = x.shape
    if c <= 8:
        return ops.nchw_to_nhwc_bf16(x, pitch)
    out = torch.zeros(n, h, w, pitch, dtype=ACT, device=x.device) if pitch != c else \
        torch.empty(n, h, w, pitch, dtype=ACT, device=x.device)
    out[..., :c].copy_(x.permute(0, 2, 3, 1))
    return out


_PLAN_CACHE: Dict[Any, Any] = {}      # (weight identity / version, input shape) -> bound plan; small LRU
_PLAN_CACHE_MAX = 96


def conv_forward(x: Tensor, weight: Tensor, bias: Optional[Tensor], stride: int, transposed: bool,
                 tap_mask: int = 0) -> Tensor:
    """One conv()/deconv()/MaskedConv2d on the tensor-core kernel, NCHW fp32 in and out: the implementation of
    `torch.ops.masic_b200.conv2d`.  Module-granularity (unfused) execution, used when the reference's own MASIC.py
    drives the layers one by one.  Plans (packed weights + bound staging buffers) are cached per (weight, bias, input
    shape) and rebuilt when either tensor's version or storage changes."""
    if not x.is_cuda:
        raise MasicError("masic_b200 conv: CUDA tensors only (no CPU fallback)")
    k = weight.shape[-1]
    s = int(stride)
    cin, cout = (weight.shape[0], weight.shape[1]) if transposed else (weight.shape[1], weight.shape[0])
    if max(cin, cout) <= 8:               # tiny-channel layers: CUDA-core direct conv
        if transposed and s != 1:
            raise MasicError("tiny transposed conv with stride 2 is not on MASIC's path")
        return ops.conv_small(x, None, weight, bias, ksize=k, stride=s, transposed_s1=transposed)
    key = (tuple(x.shape), x.device, weight.data_ptr(), weight._version, s, bool(transposed), int(tap_mask),
           None if bias is None else (bias.data_ptr(), bias._version))
    ent = _PLAN_CACHE.get(key)
    if ent is None:
        if len(_PLAN_CACHE) >= _PLAN_CACHE_MAX:
            _PLAN_CACHE.pop(next(iter(_PLAN_CACHE)))
        n, _, h, w = x.shape
        cin_p = max(16, -(-cin // 16) * 16)
        wt = weight.detach().float()
        if cin_p != cin:
            pad_shape = list(wt.shape)
            pad_shape[0 if transposed else 1] = cin_p
            wp = torch.zeros(pad_shape, device=wt.device)
            if transposed:
                wp[:cin] = wt
            else:
                wp[:, :cin] = wt
            wt = wp
        xin = torch.empty(n, h, w, cin_p, dtype=ACT, device=x.device)
        if transposed and s == 2:
            if cout <= 8:
                kind, n_tile = DECONV_S2_SUBPIX, 16
            else:
                kind, n_tile = DECONV_S2, (128 if cout % 128 == 0 else 192 if cout % 192 == 0 else 64)
        else:
            kind, n_tile = CONV, (128 if cout % 128 == 0 else 192 if cout % 192 == 0 else 64)
        packed = PackedConv(kind=kind, ksize=k, c_in=cin_p, c_out=cout, n_tile=n_tile, weight=wt,
                            transposed=transposed, bias=bias, f16=F16)
        if kind == DECONV_S2:
            ho, wo = 2 * h, 2 * w
        elif kind == CONV and s == 2:
            ho, wo = h // 2, w // 2
        else:
            ho, wo = h, w
        out = torch.empty(n, ho, wo, packed.c_out_pad, dtype=torch.float32, device=x.device)
        plan = ConvPlan(packed=packed, stride=s if kind == CONV else 1, tap_mask=tap_mask, x=xin, out=out)
        ent = _PLAN_CACHE[key] = (plan, xin, out, kind, cin_p)
    plan, xin, out, kind, cin_p = ent
    n, c, h, w = x.shape
    if c <= 8:
        ops.nchw_to_nhwc_bf16(x, cin_p, out=xin)
    else:
        if cin_p != c:
            xin.zero_()
        xin[..., :c].copy_(x.permute(0, 2, 3, 1))
    plan.launch()
    if kind == DECONV_S2_SUBPIX:
        res = torch.empty(n, cout, 2 * h, 2 * w, dtype=torch.float32, device=x.device)
        ops.subpix_to_nchw_into(out, res)
        return res
    return ops.nhwc_to_nchw_f32(out, cout)


class _TCConvMixin:
    """nn.Conv2d / nn.ConvTranspose2d parameter containers whose forward is `torch.ops.masic_b200.conv2d`."""

    def _tc_forward(self, x: Tensor, *, transposed: bool, tap_mask: int = 0) -> Tensor:
        _require_inference(self, x)
        from . import torch_ops  # noqa: F401  (registers torch.ops.masic_b200.*)
        return torch.ops.masic_b200.conv2d(x, self.weight, self.bias, self.stride[0], transposed, tap_mask)


class Conv2d(_TCConvMixin, nn.Conv2d):
    def forward(self, x: Tensor) -> Tensor:   # noqa: D401
        return self._tc_forward(x, transposed=False)


class ConvTranspose2d(_TCConvMixin, nn.ConvTranspose2d):
    def forward(self, x: Tensor, output_size=None) -> Tensor:
        if output_size is not None:
            want = tuple(int(v) for v in output_size)[-2:]
            s, k, p, op = self.stride[0], self.kernel_size[0], self.padding[0], self.output_padding[0]
            have = tuple((d - 1) * s - 2 * p + k + op for d in x.shape[-2:])
            if want != have:
                raise MasicError(f"ConvTranspose2d: output_size {want} differs from the size the layer's own "
                                 f"output_padding gives ({have}); only deconv()'s geometry is on the sm_100a path")
        return self._tc_forward(x, transposed=True)


def conv(in_channels, out_channels, kernel_size=5, stride=2):
    """compressai/models/utils.py:128-135."""
    return Conv2d(in_channels, out_channels, kernel_size=kernel_size, stride=stride, padding=kernel_size // 2)


def deconv(in_channels, out_channels, kernel_size=5, stride=2):
    """compressai/models/utils.py:138-146."""
    return ConvTranspose2d(in_channels, out_channels, kernel_size=kernel_size, stride=stride,
                           output_padding=stride - 1, padding=kernel_size // 2)


class MaskedConv2d(_TCConvMixin, nn.Conv2d):
    """compressai/layers/layers.py:52-78.  The reference multiplies weight.data by the mask in
    place on every forward; that side effect (visible through state_dict) is kept, and the
    kernel additionally skips the 13 dead taps of mask 'A' instead of multiplying by zero."""

    def __init__(self, *args: Any, mask_type: str = "A", **kwargs: Any):
        super().__init__(*args, **kwargs)
        if mask_type not in ("A", "B"):
            raise ValueError(f'Invalid "mask_type" value "{mask_type}"')
        self.register_buffer("mask", torch.ones_like(self.weight.data))
        _, _, h, w = self.mask.size()
        self.mask[:, :, h // 2, w // 2 + (mask_type == "B"):] = 0
        self.mask[:, :, h // 2 + 1:] = 0
        self.mask_type = mask_type

    def tap_mask(self) -> int:
        kh, kw = self.kernel_size
        m = self.mask[0, 0]
        return sum(1 << (ky * kw + kx) for ky in range(kh) for kx in range(kw) if float(m[ky, kx]) != 0.0)

    def forward(self, x: Tensor) -> Tensor:
        self.weight.data *= self.mask
        return self._tc_forward(x, transposed=False, tap_mask=self.tap_mask())


def conv3x3(in_ch: int, out_ch: int, stride: int = 1) -> nn.Module:
    """compressai/layers/layers.py:81-83."""
    return Conv2d(in_ch, out_ch, kernel_size=3, stride=stride, padding=1)


def conv1x1(in_ch: int, out_ch: int, stride: int = 1) -> nn.Module:
    return Conv2d(in_ch, out_ch, kernel_size=1, stride=stride)


class ResidualBlock(nn.Module):
    """compressai/layers/layers.py:160-190 (used by the CQE network, MASIC.py:149-164)."""

    def __init__(self, in_ch: int, out_ch: int):
        super().__init__()
        self.conv1 = conv3x3(in_ch, out_ch)
        self.leaky_relu = nn.LeakyReLU(inplace=True)
        self.conv2 = conv3x3(out_ch, out_ch)
        self.skip = conv1x1(in_ch, out_ch) if in_ch != out_ch else None

    def forward(self, x: Tensor) -> Tensor:
        identity = x
        out = self.leaky_relu(self.conv1(x))
        out = self.leaky_relu(self.conv2(out))
        if self.skip is not None:
            identity = self.skip(x)
        return out + identity


# ----------------------------------------------------------------------------- GDN
class GDN(nn.Module):
    """compressai/layers/gdn.py:41-92.  Stand-alone forward = a 1x1 tensor-core GEMM of x^2 against
    gamma' (+beta') followed by x * rsqrt(.) ; inside HSICEngine the same maths is fused into the
    producing conv's epilogue."""

    def __init__(self, in_channels: int, inverse: bool = False, beta_min: float = 1e-6, gamma_init: float = 0.1):
        super().__init__()
        beta_min = float(beta_min)
        gamma_init = float(gamma_init)
        self.inverse = bool(inverse)
        self.beta_min = beta_min
        self.beta_reparam = NonNegativeParametrizer(minimum=beta_min)
        beta = torch.ones(in_channels)
        beta = self.beta_reparam.init(beta)
        self.beta = nn.Parameter(beta)
        self.gamma_reparam = NonNegativeParametrizer()
        gamma = gamma_init * torch.eye(in_channels)
        gamma = self.gamma_reparam.init(gamma)
        self.gamma = nn.Parameter(gamma)

    def forward(self, x: Tensor) -> Tensor:
        _require_inference(self, x)
        from . import torch_ops  # noqa: F401
        return torch.ops.masic_b200.gdn(x, self.beta, self.gamma, self.inverse, self.beta_min)
