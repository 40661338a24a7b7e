"""Functional wrappers over the C ABI (include/masic_b200.h): torch tensors in, torch tensors out.

PyTorch is used for device memory and streams only; every function here launches a
hand-written CUDA kernel through libmasic_b200.so and raises if handed a CPU tensor —
there is no CPU or ATen fallback on this path.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import ACT_LEAKY, ACT_NONE, ACT_RELU, GDN_FWD, GDN_INV, GDN_NONE, MasicError, check

F16 = _lib.FMT_F16              # inference runs on fp16 operands / activations (csrc/cvt16.cuh)
ACT16 = _lib.act_dtype(F16)

SCALE_BOUND = 0.11


def _s() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need_cuda(*ts: Optional[torch.Tensor]) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise MasicError("masic_b200 ops run on CUDA tensors only (no CPU fallback); got a "
                             f"{t.device} tensor")


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


# --------------------------------------------------------------------------- entropy models
def gmm_likelihood(y: torch.Tensor, sigma: torch.Tensor, mu: torch.Tensor, weights: torch.Tensor,
                   K: int = 5, weights_are_logits: bool = False, scale_bound: float = SCALE_BOUND,
                   want_symbols: bool = False):
    """NCHW fp32 in/out.  Returns (y_hat, likelihood[, symbols])."""
    _need_cuda(y, sigma, mu, weights)
    y, sigma, mu, weights = map(_f32c, (y, sigma, mu, weights))
    n, m, h, w = y.shape
    if sigma.shape != (n, m * K, h, w) or mu.shape != sigma.shape or weights.shape != sigma.shape:
        raise ValueError("scales/means/weights must be (N, M*K, H, W)")
    y_hat = torch.empty_like(y)
    lik = torch.empty_like(y)
    sym = torch.empty(y.shape, dtype=torch.int32, device=y.device) if want_symbols else None
    check(_lib.load().masic_gmm_likelihood_fwd(
        y.data_ptr(), sigma.data_ptr(), mu.data_ptr(), weights.data_ptr(), int(weights_are_logits), 0,
        n, m, K, h * w, float(scale_bound), y_hat.data_ptr(), lik.data_ptr(), _p(sym), 0,
        None, 0, 0, None, 0, 0, F16, _s()), "masic_gmm_likelihood_fwd")
    return (y_hat, lik, sym) if want_symbols else (y_hat, lik)


def gc_likelihood(y: torch.Tensor, scales: torch.Tensor, means: Optional[torch.Tensor] = None,
                  scale_bound: float = SCALE_BOUND, want_symbols: bool = False):
    _need_cuda(y, scales, means)
    y, scales = _f32c(y), _f32c(scales)
    if means is not None:
        means = _f32c(means.expand_as(y))
    y_hat, lik = torch.empty_like(y), torch.empty_like(y)
    sym = torch.empty(y.shape, dtype=torch.int32, device=y.device) if want_symbols else None
    check(_lib.load().masic_gc_likelihood_fwd(y.data_ptr(), scales.data_ptr(), _p(means), y.numel(),
                                              float(scale_bound), y_hat.data_ptr(), lik.data_ptr(), _p(sym), _s()),
          "masic_gc_likelihood_fwd")
    return (y_hat, lik, sym) if want_symbols else (y_hat, lik)


def gc_build_indexes(scales: torch.Tensor, scale_table: torch.Tensor, scale_bound: float = SCALE_BOUND):
    _need_cuda(scales)
    scales = _f32c(scales)
    table = _f32c(scale_table.to(scales.device))
    idx = torch.empty(scales.shape, dtype=torch.int32, device=scales.device)
    check(_lib.load().masic_gc_build_indexes(scales.data_ptr(), scales.numel(), table.data_ptr(), table.numel(),
                                             float(scale_bound), idx.data_ptr(), _s()), "masic_gc_build_indexes")
    return idx


def quantize(x: torch.Tensor, means: Optional[torch.Tensor] = None, mode: str = "dequantize"):
    """EntropyModel._quantize for 'dequantize' and 'symbols' (entropy_models.py:98-125)."""
    _need_cuda(x, means)
    x = _f32c(x)
    if means is not None:
        means = _f32c(means.expand_as(x))
    if x.numel() == 0:
        return torch.empty(x.shape, dtype=torch.float32 if mode == "dequantize" else torch.int32, device=x.device)
    if mode == "dequantize":
        out = torch.empty_like(x)
        check(_lib.load().masic_quantize(x.data_ptr(), _p(means), x.numel(), out.data_ptr(), None, _s()), "masic_quantize")
        return out
    if mode == "symbols":
        out = torch.empty(x.shape, dtype=torch.int32, device=x.device)
        check(_lib.load().masic_quantize(x.data_ptr(), _p(means), x.numel(), None, out.data_ptr(), _s()), "masic_quantize")
        return out
    raise ValueError(f'Invalid quantization mode: "{mode}"')


def _ptr_array(ts: Sequence[torch.Tensor]):
    arr = (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])
    return arr


def eb_forward(z: torch.Tensor, matrices: Sequence[torch.Tensor], biases: Sequence[torch.Tensor],
               factors: Sequence[torch.Tensor], quantiles: torch.Tensor, want_symbols: bool = False,
               want_lik: bool = True):
    """EntropyBottleneck.forward in eval mode on an NCHW fp32 tensor."""
    _need_cuda(z, quantiles, *matrices)
    if len(matrices) != 5 or len(biases) != 5 or len(factors) != 4:
        raise MasicError("masic_eb_fwd supports the reference's filters=(3,3,3,3) only")
    z = _f32c(z)
    n, c, h, w = z.shape
    ms = [_f32c(t.detach()) for t in matrices]
    bs = [_f32c(t.detach()) for t in biases]
    fs = [_f32c(t.detach()) for t in factors]
    q = _f32c(quantiles.detach())
    z_hat = torch.empty_like(z)
    lik = torch.empty_like(z) if want_lik else None
    sym = torch.empty(z.shape, dtype=torch.int32, device=z.device) if want_symbols else None
    check(_lib.load().masic_eb_fwd(z.data_ptr(), 0, n, c, h * w, _ptr_array(ms), _ptr_array(bs), _ptr_array(fs),
                                   q.data_ptr(), z_hat.data_ptr(), _p(lik), _p(sym), 0, None, 0, F16, _s()), "masic_eb_fwd")
    return z_hat, lik, sym


def pmf_to_quantized_cdf(pmf: Sequence[float], precision: int = 16):
    """compressai._CXX.pmf_to_quantized_cdf (host, integer-exact)."""
    p = np.ascontiguousarray(pmf, dtype=np.float32)
    out = np.zeros(p.size + 1, dtype=np.uint32)
    rc = _lib.load().masic_pmf_to_quantized_cdf(p.ctypes.data, p.size, precision, out.ctypes.data)
    if rc == 1:
        raise ValueError("Invalid `pmf`, non-finite or negative element found")
    if rc == 2:
        raise ValueError("Invalid `pmf`: at least one element must have a non-zero probability.")
    check(rc, "masic_pmf_to_quantized_cdf")
    return [int(v) for v in out]


def pmf_table_to_cdf(pmf: torch.Tensor, tail_mass: torch.Tensor, pmf_length: torch.Tensor, max_length: int,
                     precision: int = 16) -> torch.Tensor:
    """EntropyModel._pmf_to_cdf (entropy_models.py:136-142) -> int32 (rows, max_length + 2), CPU tensor."""
    pm = np.ascontiguousarray(pmf.detach().cpu().float().numpy())
    tm = np.ascontiguousarray(tail_mass.detach().cpu().float().reshape(-1).numpy())
    ln = np.ascontiguousarray(pmf_length.detach().cpu().to(torch.int32).numpy())
    rows = pm.shape[0]
    out = np.zeros((rows, max_length + 2), dtype=np.int32)
    rc = _lib.load().masic_pmf_table_to_cdf(pm.ctypes.data, rows, pm.shape[1], tm.ctypes.data, ln.ctypes.data,
                                            int(max_length), precision, out.ctypes.data)
    if rc in (1, 2, 3):
        raise ValueError("Invalid `pmf` row while building the CDF table")
    check(rc, "masic_pmf_table_to_cdf")
    return torch.from_numpy(out)


# --------------------------------------------------------------------------- image domain
def warp_prepare(M: torch.Tensor, src_hw: Tuple[int, int], dst_hw: Tuple[int, int], invert: bool = False):
    _need_cuda(M)
    M = _f32c(M)
    T = torch.empty(M.shape, dtype=torch.float64, device=M.device)
    check(_lib.load().masic_warp_prepare(M.data_ptr(), M.shape[0], src_hw[0], src_hw[1], dst_hw[0], dst_hw[1],
                                         int(invert), T.data_ptr(), _s()), "masic_warp_prepare")
    return T


def warp_perspective(src: Optional[torch.Tensor], M: torch.Tensor, dsize: Tuple[int, int], *,
                     invert: bool = False, ones_shape: Optional[Tuple[int, int, int, int]] = None,
                     bf16_pitch: int = 0):
    """kornia.warp_perspective(src, M, dsize) (0.5.0: bilinear, zeros, align_corners=True).
    src=None with ones_shape=(N,C,H,W) warps an all-ones image (mask())."""
    _need_cuda(src, M)
    if src is not None:
        src = _f32c(src)
        n, c, h, w = src.shape
    else:
        n, c, h, w = ones_shape
    ho, wo = dsize
    T = warp_prepare(M, (h, w), (ho, wo), invert)
    dst = torch.empty(n, c, ho, wo, dtype=torch.float32, device=M.device)
    dst_bf = torch.empty(n, ho, wo, bf16_pitch, dtype=ACT16, device=M.device) if bf16_pitch else None
    check(_lib.load().masic_warp_perspective_fwd(_p(src), n, c, h, w, ho, wo, T.data_ptr(), dst.data_ptr(),
                                                 _p(dst_bf), bf16_pitch, 0, 0, F16, _s()), "masic_warp_perspective_fwd")
    return (dst, dst_bf) if bf16_pitch else dst


def conv_small(in0: torch.Tensor, in1: Optional[torch.Tensor], weight: torch.Tensor, bias: Optional[torch.Tensor],
               *, ksize: int, stride: int, transposed_s1: bool = False, act: int = ACT_NONE, gdn: int = GDN_NONE,
               beta: Optional[torch.Tensor] = None, gamma: Optional[torch.Tensor] = None, beta_min: float = 1e-6,
               out: Optional[torch.Tensor] = None, out_bf16: Optional[torch.Tensor] = None):
    _need_cuda(in0, in1, weight)
    in0 = _f32c(in0)
    in1 = None if in1 is None else _f32c(in1)
    n, c0, h, w = in0.shape
    c1 = 0 if in1 is None else in1.shape[1]
    weight = _f32c(weight.detach())
    c_out = weight.shape[1] if transposed_s1 else weight.shape[0]
    bias = None if bias is None else _f32c(bias.detach())
    beta = None if beta is None else _f32c(beta.detach())
    gamma = None if gamma is None else _f32c(gamma.detach())
    ho, wo = -(-h // stride), -(-w // stride)
    if out is None and out_bf16 is None:
        out = torch.empty(n, c_out, ho, wo, dtype=torch.float32, device=in0.device)
    check(_lib.load().masic_conv_small_nchw(in0.data_ptr(), c0, _p(in1), c1, n, h, w, weight.data_ptr(),
                                            int(transposed_s1), _p(bias), c_out, ksize, stride, act, gdn, _p(beta),
                                            _p(gamma), float(beta_min), _p(out), _p(out_bf16),
                                            0 if out_bf16 is None else out_bf16.shape[3], 0, 0, F16, _s()),
          "masic_conv_small_nchw")
    return out if out is not None else out_bf16


def mask2weights(mask: torch.Tensor, weights, biases, nhwc_out: bool = False):
    """mask2weights.forward (MASIC.py:472-506) in one launch.  weights / biases: the four conv3x3 stride-2 layers'
    parameters (maskconv.0, .2, .4, .6).  Returns the (n,3,h/16,w/16) softmax weights (and the NHWC copy)."""
    _need_cuda(mask, *weights)
    mask = _f32c(mask)
    n, c, h, w = mask.shape
    if c != 1 or len(weights) != 4 or len(biases) != 4:
        raise MasicError("mask2weights: mask must be (n,1,h,w) with four layers of parameters")
    shapes = [(3, 1, 3, 3), (6, 3, 3, 3), (6, 6, 3, 3), (3, 6, 3, 3)]
    ws = [_f32c(t.detach()) for t in weights]
    for t, shp in zip(ws, shapes):
        if tuple(t.shape) != shp:
            raise MasicError(f"mask2weights: weight shape {tuple(t.shape)} != {shp}")
    bs = [None if t is None else _f32c(t.detach()) for t in biases]
    ho, wo = h, w
    for _ in range(4):
        ho, wo = (ho + 1) // 2, (wo + 1) // 2
    out = torch.empty(n, 3, ho, wo, dtype=torch.float32, device=mask.device)
    out_nhwc = torch.empty(n, ho, wo, 3, dtype=torch.float32, device=mask.device) if nhwc_out else None
    check(_lib.load().masic_mask2weights(mask.data_ptr(), n, h, w, ws[0].data_ptr(), _p(bs[0]), ws[1].data_ptr(), _p(bs[1]),
                                         ws[2].data_ptr(), _p(bs[2]), ws[3].data_ptr(), _p(bs[3]), out.data_ptr(),
                                         _p(out_nhwc), _s()), "masic_mask2weights")
    return (out, out_nhwc) if nhwc_out else out


def softmax_channels(x: torch.Tensor, nhwc_out: bool = False):
    _need_cuda(x)
    x = _f32c(x)
    n, c, h, w = x.shape
    o1 = torch.empty_like(x)
    o2 = torch.empty(n, h, w, c, dtype=torch.float32, device=x.device) if nhwc_out else None
    check(_lib.load().masic_softmax_channels(x.data_ptr(), n, c, h * w, o1.data_ptr(), _p(o2), _s()),
          "masic_softmax_channels")
    return (o1, o2) if nhwc_out else o1


def nchw_to_nhwc_bf16(x: torch.Tensor, pitch: int, out: Optional[torch.Tensor] = None):
    _need_cuda(x)
    x = _f32c(x)
    n, c, h, w = x.shape
    if out is None:
        out = torch.empty(n, h, w, pitch, dtype=ACT16, device=x.device)
    check(_lib.load().masic_nchw_to_nhwc_bf16(x.data_ptr(), n, c, h, w, out.data_ptr(), pitch, 0, 0, F16, _s()),
          "masic_nchw_to_nhwc_bf16")
    return out


def nhwc_to_nchw_f32(x: torch.Tensor, c: Optional[int] = None, out: Optional[torch.Tensor] = None):
    _need_cuda(x)
    assert x.dtype == torch.float32 and x.is_contiguous()
    n, h, w, pitch = x.shape
    c = c or pitch
    if out is None:
        out = torch.empty(n, c, h, w, dtype=torch.float32, device=x.device)
    check(_lib.load().masic_nhwc_to_nchw_f32(x.data_ptr(), n, c, h * w, pitch, out.data_ptr(), _s()),
          "masic_nhwc_to_nchw_f32")
    return out


# --------------------------------------------------------------------------- image quality
MS_SSIM_WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)     # pytorch_msssim's default level weights


def ssim_per_channel(x: torch.Tensor, y: torch.Tensor, data_range: float, weights: Sequence[float],
                     k: Tuple[float, float] = (0.01, 0.03), nonneg_last: bool = True) -> torch.Tensor:
    """The (N, C) per-channel values of pytorch_msssim 1.0 on (N, C, H, W) fp32 CUDA tensors (csrc/msssim.cu):
    len(weights) levels; ms_ssim is 5 levels with nonneg_last=True, ssim is weights=(1.0,)."""
    _need_cuda(x, y)
    if x.dtype != torch.float32 or y.dtype != torch.float32:
        raise MasicError("masic_ms_ssim runs on float32 images only")
    if x.dim() != 4 or x.shape != y.shape:
        raise ValueError(f"ms_ssim needs two (N, C, H, W) tensors of one shape, got {tuple(x.shape)} and {tuple(y.shape)}")
    x, y = x.contiguous(), y.contiguous()
    n, c, h, w = x.shape
    lib = _lib.load()
    levels = len(weights)
    nbytes = lib.masic_ms_ssim_scratch_bytes(n, c, h, w, levels)
    check(min(int(nbytes), 0), f"masic_ms_ssim_scratch_bytes ({levels} levels of {h}x{w} need >= 11x11 each)")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    out = torch.empty(n, c, dtype=torch.float32, device=x.device)
    wts = (C.c_float * levels)(*map(float, weights))
    check(lib.masic_ms_ssim(x.data_ptr(), y.data_ptr(), n, c, h, w, levels, float(data_range), float(k[0]), float(k[1]),
                            wts, int(nonneg_last), scratch.data_ptr(), out.data_ptr(), _s()), "masic_ms_ssim")
    return out


def ms_ssim(x: torch.Tensor, y: torch.Tensor, data_range: float = 255, size_average: bool = True,
            weights: Optional[Sequence[float]] = None, k: Tuple[float, float] = (0.01, 0.03)) -> torch.Tensor:
    """pytorch_msssim.ms_ssim (1.0): the mean over (N, C), or over C only (shape (N,)) with size_average=False."""
    v = ssim_per_channel(x, y, data_range, MS_SSIM_WEIGHTS if weights is None else weights, k, True)
    return v.mean() if size_average else v.mean(1)


def ssim(x: torch.Tensor, y: torch.Tensor, data_range: float = 255, size_average: bool = True,
         k: Tuple[float, float] = (0.01, 0.03), nonnegative_ssim: bool = False) -> torch.Tensor:
    """pytorch_msssim.ssim (1.0): single-scale SSIM, relu'd per channel with nonnegative_ssim=True."""
    v = ssim_per_channel(x, y, data_range, (1.0,), k, nonnegative_ssim)
    return v.mean() if size_average else v.mean(1)
