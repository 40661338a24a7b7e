"""`torch.library` registration of the C-ABI kernels (the "thin C-ABI torch custom-op extension" of the north-star,
SURVEY §8(b)): every op below is a `torch.ops.masic_b200.*` custom op whose CUDA implementation is one call (or a short
fixed sequence of calls) into libmasic_b200.so, with a fake (meta) implementation for shape inference, so the ops are
visible to the dispatcher, `torch.compile` / `torch.export` tracing and `torch.library.opcheck`.  The nn.Modules of
masic_b200.layers / entropy_models call these ops; the fused engine (engine.py) calls the C ABI directly.

There is no CPU implementation: dispatching one of these ops on CPU tensors raises.  None of them registers an
autograd formula (inference ops; the training step is the fused HSICTrainer), so differentiating through one raises
PyTorch's "not differentiable" error instead of silently returning zeros.

    torch.ops.masic_b200.conv2d(x, weight, bias, stride, transposed, tap_mask) -> Tensor      conv()/deconv()/MaskedConv2d
    torch.ops.masic_b200.gdn(x, beta, gamma, inverse, beta_min) -> Tensor                      GDN.forward
    torch.ops.masic_b200.warp_perspective(src, M, h_out, w_out) -> Tensor                      kornia.warp_perspective
    torch.ops.masic_b200.gmm_likelihood(y, scales, means, weights, scale_bound) -> (y_hat, lik)
    torch.ops.masic_b200.gc_likelihood(y, scales, means, scale_bound) -> (y_hat, lik)
    torch.ops.masic_b200.gc_build_indexes(scales, scale_table, scale_bound) -> Tensor(int32)
    torch.ops.masic_b200.quantize(x, means, symbols) -> Tensor
    torch.ops.masic_b200.eb_forward(z, matrices, biases, factors, quantiles) -> (z_hat, lik)
    torch.ops.masic_b200.ms_ssim(x, y, data_range, weights, k1, k2, nonneg_last) -> Tensor(N, C)  pytorch_msssim
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch
from torch import Tensor

from . import ops
from ._lib import MasicError

NS = "masic_b200"


def _cuda_only(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise MasicError("torch.ops.masic_b200.* run on CUDA tensors only (no CPU fallback)")


# ----------------------------------------------------------------------------- conv / deconv / masked conv
@torch.library.custom_op(f"{NS}::conv2d", mutates_args=(), device_types="cuda")
def conv2d(x: Tensor, weight: Tensor, bias: Optional[Tensor], stride: int, transposed: bool, tap_mask: int) -> Tensor:
    """nn.Conv2d(k, stride, padding=k//2) / nn.ConvTranspose2d(k, stride, padding=k//2, output_padding=stride-1) of
    compressai/models/utils.py:128-146 on NCHW fp32 tensors; tap_mask != 0 keeps only the listed taps (MaskedConv2d)."""
    from .layers import conv_forward
    return conv_forward(x, weight, bias, stride, transposed, tap_mask)


@conv2d.register_fake
def _(x, weight, bias, stride, transposed, tap_mask):
    n, _, h, w = x.shape
    cout = weight.shape[1] if transposed else weight.shape[0]
    if transposed:
        ho, wo = h * stride, w * stride
    else:
        ho, wo = -(-h // stride), -(-w // stride)
    return x.new_empty((n, cout, ho, wo), dtype=torch.float32)


# ----------------------------------------------------------------------------- GDN
@torch.library.custom_op(f"{NS}::gdn", mutates_args=(), device_types="cuda")
def gdn(x: Tensor, beta: Tensor, gamma: Tensor, inverse: bool, beta_min: float) -> Tensor:
    """compressai/layers/gdn.py:77-92 with the stored (re-parametrised) beta / gamma."""
    _cuda_only(x, beta, gamma)
    x = x.float().contiguous()
    out = torch.empty_like(x)
    ops.gdn_nchw_into(x, beta.detach().float().contiguous(), gamma.detach().float().contiguous(), out, inverse=inverse,
                      beta_min=beta_min)
    return out


@gdn.register_fake
def _(x, beta, gamma, inverse, beta_min):
    return torch.empty_like(x, dtype=torch.float32)


# ----------------------------------------------------------------------------- warp
@torch.library.custom_op(f"{NS}::warp_perspective", mutates_args=(), device_types="cuda")
def warp_perspective(src: Tensor, M: Tensor, h_out: int, w_out: int) -> Tensor:
    """kornia.warp_perspective(src, M, (h_out, w_out)) — bilinear, zeros, align_corners=True (kornia 0.5.0)."""
    _cuda_only(src, M)
    return ops.warp_perspective(src, M, (h_out, w_out))


@warp_perspective.register_fake
def _(src, M, h_out, w_out):
    return src.new_empty((src.shape[0], src.shape[1], h_out, w_out), dtype=torch.float32)


# ----------------------------------------------------------------------------- entropy models
@torch.library.custom_op(f"{NS}::gmm_likelihood", mutates_args=(), device_types="cuda")
def gmm_likelihood(y: Tensor, scales: Tensor, means: Tensor, weights: Tensor, scale_bound: float) -> Tuple[Tensor, Tensor]:
    """GaussianMixtureConditional_gf.forward (eval), entropy_models.py:849-858: (round(y), mixture likelihood)."""
    _cuda_only(y, scales, means, weights)
    k = scales.shape[1] // y.shape[1]
    return ops.gmm_likelihood(y, scales, means, weights, K=k, weights_are_logits=False, scale_bound=scale_bound)


@gmm_likelihood.register_fake
def _(y, scales, means, weights, scale_bound):
    return torch.empty_like(y, dtype=torch.float32), torch.empty_like(y, dtype=torch.float32)


@torch.library.custom_op(f"{NS}::gc_likelihood", mutates_args=(), device_types="cuda")
def gc_likelihood(y: Tensor, scales: Tensor, means: Optional[Tensor], scale_bound: float) -> Tuple[Tensor, Tensor]:
    """GaussianConditional.forward (eval), entropy_models.py:546-554."""
    _cuda_only(y, scales, means)
    return ops.gc_likelihood(y, scales, means, scale_bound)


@gc_likelihood.register_fake
def _(y, scales, means, scale_bound):
    return torch.empty_like(y, dtype=torch.float32), torch.empty_like(y, dtype=torch.float32)


@torch.library.custom_op(f"{NS}::gc_build_indexes", mutates_args=(), device_types="cuda")
def gc_build_indexes(scales: Tensor, scale_table: Tensor, scale_bound: float) -> Tensor:
    """GaussianConditional.build_indexes, entropy_models.py:556-562 (int32 CDF indexes)."""
    _cuda_only(scales)
    return ops.gc_build_indexes(scales, scale_table, scale_bound)


@gc_build_indexes.register_fake
def _(scales, scale_table, scale_bound):
    return torch.empty_like(scales, dtype=torch.int32)


@torch.library.custom_op(f"{NS}::quantize", mutates_args=(), device_types="cuda")
def quantize(x: Tensor, means: Optional[Tensor], symbols: bool) -> Tensor:
    """EntropyModel._quantize, entropy_models.py:98-125: 'symbols' (int32) or 'dequantize' (fp32)."""
    _cuda_only(x, means)
    return ops.quantize(x, means, "symbols" if symbols else "dequantize")


@quantize.register_fake
def _(x, means, symbols):
    return torch.empty_like(x, dtype=torch.int32 if symbols else torch.float32)


@torch.library.custom_op(f"{NS}::eb_forward", mutates_args=(), device_types="cuda")
def eb_forward(z: Tensor, matrices: List[Tensor], biases: List[Tensor], factors: List[Tensor],
               quantiles: Tensor) -> Tuple[Tensor, Tensor]:
    """EntropyBottleneck.forward (eval), entropy_models.py:384-411."""
    _cuda_only(z, quantiles)
    z_hat, lik, _ = ops.eb_forward(z, matrices, biases, factors, quantiles)
    return z_hat, lik


@eb_forward.register_fake
def _(z, matrices, biases, factors, quantiles):
    return torch.empty_like(z, dtype=torch.float32), torch.empty_like(z, dtype=torch.float32)


# ----------------------------------------------------------------------------- image quality
@torch.library.custom_op(f"{NS}::ms_ssim", mutates_args=(), device_types="cuda")
def ms_ssim(x: Tensor, y: Tensor, data_range: float, weights: List[float], k1: float, k2: float,
            nonneg_last: bool) -> Tensor:
    """pytorch_msssim 1.0 per (n, c): ms_ssim with the 5 level weights (nonneg_last=True), ssim with weights=[1.0]
    (nonneg_last = nonnegative_ssim).  The reference's eval loop reports it per pair, test2_real.py:88-114."""
    _cuda_only(x, y)
    return ops.ssim_per_channel(x, y, data_range, weights, (k1, k2), nonneg_last)


@ms_ssim.register_fake
def _(x, y, data_range, weights, k1, k2, nonneg_last):
    return x.new_empty((x.shape[0], x.shape[1]), dtype=torch.float32)


OPS = ("conv2d", "gdn", "warp_perspective", "gmm_likelihood", "gc_likelihood", "gc_build_indexes", "quantize", "eb_forward",
       "ms_ssim")
