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
    if t is None:
        return None
    if not t.is_cuda:
        raise MasicError("masic_b200 kernels need CUDA tensors (no CPU fallback)")
    return t.data_ptr()


def _ptr_array(ts: Sequence[Optional[torch.Tensor]]):
    return (C.c_void_p * len(ts))(*[_p(t) for t in ts])


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
# The `*_into` launchers write caller-owned tensors on the current stream, sizes, row layouts and 16-bit formats taken
# from the tensors.  They run during CUDA-graph capture, where a temporary would go stale, so they allocate and convert
# nothing: a CPU, non-contiguous, wrong-dtype or wrongly shaped tensor raises MasicError before anything is launched.
_F32, _F64, _HALF = (torch.float32,), (torch.float64,), (torch.float16, torch.bfloat16)
_FMT16 = {torch.float16: _lib.FMT_F16, torch.bfloat16: _lib.FMT_BF16}


def _arg(t: Optional[torch.Tensor], dtypes, shape=None) -> Optional[int]:
    """t's device pointer (None stays None) once t can be handed to the kernel as it is."""
    if t is None:
        return None
    if not t.is_cuda:
        raise MasicError(f"masic_b200 kernels need CUDA tensors (no CPU fallback); got a {t.device} tensor")
    if t.dtype not in dtypes:
        raise MasicError(f"got a {t.dtype} tensor where the kernel reads {' or '.join(map(str, dtypes))}")
    if not t.is_contiguous():
        raise MasicError("the kernel needs a contiguous tensor")
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise MasicError(f"got a tensor of shape {tuple(t.shape)} where the kernel needs {tuple(shape)}")
    return t.data_ptr()


def _img16(t: Optional[torch.Tensor], n: int, h: int, w: int, split: bool = False):
    """(pointer, pitch, row_pixels, xoff, format) of a 16-bit NHWC image (n, h, R, pitch): R == w is dense, R == w +
    IMG_XPAD padded (pixel x at column x + IMG_XOFF).  split=True stores [hi | lo] pixels (the engine's g_a_conv1 input)."""
    if t is None:
        return None, 0, 0, 0, 0
    ptr = _arg(t, _HALF)
    if t.dim() != 4 or tuple(t.shape[:2]) != (n, h) or t.shape[2] not in (w, w + _lib.IMG_XPAD):
        raise MasicError(f"a 16-bit image must be ({n}, {h}, {w} or {w} + IMG_XPAD, pitch), got {tuple(t.shape)}")
    padded = t.shape[2] != w
    return (ptr, t.shape[3], t.shape[2] if padded else 0, _lib.IMG_XOFF if padded else 0,
            _FMT16[t.dtype] | (_lib.FMT_SPLIT if split else 0))


def _launch(name: str, *args) -> None:
    check(getattr(_lib.load(), name)(*args, _s()), name)


def warp_prepare_into(M: torch.Tensor, T: torch.Tensor, src_hw: Tuple[int, int], dst_hw: Tuple[int, int],
                      invert: bool = False) -> None:
    """T (n,3,3) fp64 <- the transform the warp kernel reads for the (n,3,3) fp32 homographies M (or their inverses)."""
    n = M.shape[0]
    _launch("masic_warp_prepare", _arg(M, _F32, (n, 3, 3)), n, *src_hw, *dst_hw, int(invert), _arg(T, _F64, (n, 3, 3)))


def warp_perspective_into(src: Optional[torch.Tensor], T: torch.Tensor, dsize: Tuple[int, int], *, src_shape=None,
                          dst=None, dst16=None, split: bool = False, dst2=None, dst2_coff: int = 0, ones=None) -> None:
    """src (NCHW fp32; None: all ones of src_shape) warped by T to dsize into dst (NCHW fp32), dst16, dst2 (16-bit NHWC;
    dst2's channels at dst2_coff, the rest of the pixel untouched) and ones (the all-ones image warped, (n,1,h,w))."""
    n, c, h, w = src.shape if src is not None else src_shape
    ho, wo = dsize
    p16, pitch, row, xoff, fmt = _img16(dst16, n, ho, wo, split)
    p2, pitch2, row2, xoff2, fmt2 = _img16(dst2, n, ho, wo)
    if dst2 is not None and not row2:
        row2 = wo                  # the second destination's rows are always given: row_pixels = 0 is not "dense" there
    _launch("masic_warp_perspective_fwd", _arg(src, _F32), n, c, h, w, ho, wo, _arg(T, _F64, (n, 3, 3)),
            _arg(dst, _F32, (n, c, ho, wo)), p16, pitch, row, xoff, fmt, p2, pitch2, row2, xoff2, dst2_coff, fmt2,
            _arg(ones, _F32, (n, 1, ho, wo)))


def conv_small_into(in0: torch.Tensor, in1: Optional[torch.Tensor], weight: torch.Tensor, bias: Optional[torch.Tensor],
                    *, ksize: int, stride: int, transposed_s1: bool = False, act: int = ACT_NONE, gdn: int = GDN_NONE,
                    beta=None, gamma=None, beta_min: float = 1e-6, out=None, out16=None, split: bool = False) -> None:
    """Tiny-channel conv of cat(in0, in1) (NCHW fp32) into out (NCHW fp32) and / or out16 (16-bit NHWC)."""
    n, c0, h, w = in0.shape
    c1 = 0 if in1 is None else in1.shape[1]
    c_out = weight.shape[1] if transposed_s1 else weight.shape[0]
    ho, wo = -(-h // stride), -(-w // stride)
    _launch("masic_conv_small_nchw", _arg(in0, _F32), c0, _arg(in1, _F32, (n, c1, h, w)), c1, n, h, w,
            _arg(weight, _F32), int(transposed_s1), _arg(bias, _F32, (c_out,)), c_out, ksize, stride, act, gdn,
            _arg(beta, _F32), _arg(gamma, _F32), float(beta_min), _arg(out, _F32, (n, c_out, ho, wo)),
            *_img16(out16, n, ho, wo, split))


def nchw_to_nhwc_into(x: torch.Tensor, out: torch.Tensor, *, split: bool = False) -> None:
    """NCHW fp32 (c <= 8) -> the 16-bit NHWC image out, channels beyond c zeroed."""
    n, c, h, w = x.shape
    _launch("masic_nchw_to_nhwc_bf16", _arg(x, _F32), n, c, h, w, *_img16(out, n, h, w, split))


def nhwc_to_nchw_into(x: torch.Tensor, out: torch.Tensor) -> None:
    """The first out.shape[1] channels of the NHWC fp32 x -> NCHW fp32 out."""
    n, h, w, pitch = x.shape
    c = out.shape[1]
    _launch("masic_nhwc_to_nchw_f32", _arg(x, _F32), n, c, h * w, pitch, _arg(out, _F32, (n, c, h, w)))


def subpix_to_nchw_into(x: torch.Tensor, out: torch.Tensor) -> None:
    """A MASIC_DECONV_S2_SUBPIX plan's output (n, h, w, pitch) fp32 -> the NCHW fp32 image out (n, 3, 2h, 2w)."""
    n, h, w, pitch = x.shape
    _launch("masic_subpix_to_nchw", _arg(x, _F32), n, h, w, pitch, GDN_NONE, None, None, 1e-6,
            _arg(out, _F32, (n, 3, 2 * h, 2 * w)), None, 0, 0)


def softmax_channels_into(x: torch.Tensor, out=None, out_nhwc=None) -> None:
    """Softmax over the channels of the NCHW fp32 x into out (NCHW) and / or out_nhwc."""
    n, c, h, w = x.shape
    _launch("masic_softmax_channels", _arg(x, _F32), n, c, h * w, _arg(out, _F32, (n, c, h, w)),
            _arg(out_nhwc, _F32, (n, h, w, c)))


def mask2weights_into(mask: torch.Tensor, weights: Sequence[torch.Tensor], biases: Sequence[Optional[torch.Tensor]],
                      out=None, out_nhwc=None) -> None:
    """mask2weights.forward (MASIC.py:472-506) of the (n,1,h,w) mask into out (n,3,h/16,w/16) and / or out_nhwc."""
    n, _, h, w = mask.shape
    ho, wo = -(-h // 16), -(-w // 16)          # four stride-2 layers, each rounding up
    params = [_arg(t, _F32) for wb in zip(weights, biases) for t in wb]
    _launch("masic_mask2weights", _arg(mask, _F32, (n, 1, h, w)), n, h, w, *params, _arg(out, _F32, (n, 3, ho, wo)),
            _arg(out_nhwc, _F32, (n, ho, wo, 3)))


def gdn_nchw_into(x: torch.Tensor, beta: torch.Tensor, gamma: torch.Tensor, out: torch.Tensor, *,
                  inverse: bool = False, beta_min: float = 1e-6) -> None:
    """GDN / IGDN over the channels of the NCHW fp32 x with the stored (re-parametrised) beta (c,) and gamma (c, c)."""
    n, c, h, w = x.shape
    _launch("masic_gdn_nchw", _arg(x, _F32), n, c, h * w, _arg(beta, _F32, (c,)), _arg(gamma, _F32, (c, c)),
            float(beta_min), int(inverse), _arg(out, _F32, (n, c, h, w)))


def cqe_mask_weights_into(mask: torch.Tensor, weights: Sequence[torch.Tensor], biases: Sequence[torch.Tensor], out) -> None:
    """mask2weights_EN.forward (MASIC.py:1411-1434) of the (n,1,h,w) mask into out (n,kw,h,w)."""
    n, _, h, w = mask.shape
    kw = out.shape[1]
    ws = (C.c_void_p * 4)(*[_arg(t, _F32) for t in weights])
    bs = (C.c_void_p * 4)(*[_arg(t, _F32) for t in biases])
    _launch("masic_cqe_mask_weights", _arg(mask, _F32, (n, 1, h, w)), n, h, w, ws, bs, kw, _arg(out, _F32, (n, kw, h, w)))


def cqe_blend_images_into(a: torch.Tensor, b: torch.Tensor, weights: torch.Tensor, out: torch.Tensor) -> None:
    """MASIC.py:1470-1471: out (n,h,w,16) 16-bit = [a * weights[:,0] | b * weights[:,1] | 0] of the NCHW fp32 images."""
    n, _, h, w = b.shape
    _launch("masic_cqe_blend_images", _arg(a, _F32, (n, 3, h, w)), _arg(b, _F32, (n, 3, h, w)),
            _arg(weights, _F32, (n, 2, h, w)), n, h, w, _arg(out, _HALF, (n, h, w, 16)), _FMT16[out.dtype])


def cqe_feature_fuse_into(self_: torch.Tensor, other: torch.Tensor, weights: torch.Tensor, T: torch.Tensor,
                          out: torch.Tensor) -> None:
    """MASIC.py:1479-1482 on 16-bit NHWC maps, c = self_.shape[3]: out[..., :2c] = [self_ * w1 | warp(other, T) * w0]."""
    n, h, w, c = self_.shape
    p_out = _arg(out, _HALF)
    _launch("masic_cqe_feature_fuse", _arg(self_, (out.dtype,)), c, _arg(other, (out.dtype,)), other.shape[3], c,
            _arg(weights, _F32, (n, 2, h, w)), _arg(T, _F64, (n, 3, 3)), n, h, w, p_out, out.shape[3], _FMT16[out.dtype])


def cqe_residual_image_into(conv_out: torch.Tensor, identity: torch.Tensor, out: torch.Tensor) -> None:
    """MASIC.py:1495-1496: out (NCHW fp32) = the first 3 channels of the NHWC fp32 conv_out + identity (NCHW fp32)."""
    n, h, w, pitch = conv_out.shape
    _launch("masic_cqe_residual_image", _arg(conv_out, _F32), pitch, _arg(identity, _F32, (n, 3, h, w)), n, h, w,
            _arg(out, _F32, (n, 3, h, w)))


def pad_image_into(src: torch.Tensor, dst: torch.Tensor, top: int, left: int, unpadded=None) -> None:
    """src (n,c,h,w) uint8 (ToTensor's x / 255) or fp32 -> dst (n,c,hp,wp) fp32 zero-padded, src at (top, left), every
    element of dst written; unpadded (n,c,h,w) fp32, if given, receives the converted src from the same pass."""
    n, c, h, w = src.shape
    hp, wp = dst.shape[2:]
    _launch("masic_pad_image", _arg(src, (torch.uint8, torch.float32)), int(src.dtype == torch.uint8), n, c, h, w, hp,
            wp, top, left, _arg(dst, _F32, (n, c, hp, wp)), _arg(unpadded, _F32, (n, c, h, w)))


def homography_pad_into(h: torch.Tensor, out: torch.Tensor, top: int, left: int) -> None:
    """out (n,3,3) fp32 <- T h T^-1 for the (n,3,3) fp32 homographies h, T the translation by (left, top)."""
    n = h.shape[0]
    _launch("masic_homography_pad", _arg(h, _F32, (n, 3, 3)), n, top, left, _arg(out, _F32, (n, 3, 3)))


def rd_metrics_scratch(device) -> torch.Tensor:
    """The device scratch rd_metrics_into needs (allocate it once, outside graph capture)."""
    return torch.empty(_lib.load().masic_rd_metrics_scratch_bytes() // 8, dtype=torch.float64, device=device)


def rd_metrics_into(liks: Sequence[Optional[torch.Tensor]], x1_hat: torch.Tensor, x1: torch.Tensor,
                    x2_hat: torch.Tensor, x2: torch.Tensor, lmbda: float, scratch: torch.Tensor,
                    out: torch.Tensor) -> None:
    """RateDistortionLoss.forward into out (8 fp32, see masic_rd_metrics); a None likelihood tensor is skipped."""
    n, c, h, w = x1_hat.shape
    lp = (C.c_void_p * 4)(*[_arg(t, _F32) for t in liks])
    ln = (C.c_int64 * 4)(*[0 if t is None else t.numel() for t in liks])
    imgs = [_arg(t, _F32, (n, c, h, w)) for t in (x1_hat, x1, x2_hat, x2)]
    _launch("masic_rd_metrics", lp, ln, *imgs, n, c, h, w, float(lmbda), _arg(scratch, _F64), _arg(out, _F32, (8,)))


def warp_prepare(M: torch.Tensor, src_hw: Tuple[int, int], dst_hw: Tuple[int, int], invert: bool = False):
    M = _f32c(M)
    T = torch.empty(M.shape, dtype=torch.float64, device=M.device)
    warp_prepare_into(M, T, src_hw, dst_hw, invert)
    return T


def warp_perspective(src: Optional[torch.Tensor], M: torch.Tensor, dsize: Tuple[int, int], *,
                     invert: bool = False, ones_shape: Optional[Tuple[int, int, int, int]] = None,
                     bf16_pitch: int = 0):
    """kornia.warp_perspective(src, M, dsize) (0.5.0: bilinear, zeros, align_corners=True).
    src=None with ones_shape=(N,C,H,W) warps an all-ones image (mask())."""
    if src is not None:
        src = _f32c(src)
    n, c, h, w = src.shape if src is not None else ones_shape
    ho, wo = dsize
    T = warp_prepare(M, (h, w), (ho, wo), invert)
    dst = torch.empty(n, c, ho, wo, dtype=torch.float32, device=M.device)
    dst_bf = torch.empty(n, ho, wo, bf16_pitch, dtype=ACT16, device=M.device) if bf16_pitch else None
    warp_perspective_into(src, T, dsize, src_shape=(n, c, h, w), dst=dst, dst16=dst_bf)
    return (dst, dst_bf) if bf16_pitch else dst


def conv_small(in0: torch.Tensor, in1: Optional[torch.Tensor], weight: torch.Tensor, bias: Optional[torch.Tensor],
               *, ksize: int, stride: int, transposed_s1: bool = False, act: int = ACT_NONE, gdn: int = GDN_NONE,
               beta: Optional[torch.Tensor] = None, gamma: Optional[torch.Tensor] = None, beta_min: float = 1e-6,
               out: Optional[torch.Tensor] = None, out_bf16: Optional[torch.Tensor] = None):
    in0 = _f32c(in0)
    in1 = None if in1 is None else _f32c(in1)
    n, _, h, w = in0.shape
    weight = _f32c(weight.detach())
    c_out = weight.shape[1] if transposed_s1 else weight.shape[0]
    bias = None if bias is None else _f32c(bias.detach())
    beta = None if beta is None else _f32c(beta.detach())
    gamma = None if gamma is None else _f32c(gamma.detach())
    ho, wo = -(-h // stride), -(-w // stride)
    if out is None and out_bf16 is None:
        out = torch.empty(n, c_out, ho, wo, dtype=torch.float32, device=in0.device)
    conv_small_into(in0, in1, weight, bias, ksize=ksize, stride=stride, transposed_s1=transposed_s1, act=act, gdn=gdn,
                    beta=beta, gamma=gamma, beta_min=beta_min, out=out, out16=out_bf16)
    return out if out is not None else out_bf16


def mask2weights(mask: torch.Tensor, weights, biases, nhwc_out: bool = False):
    """mask2weights.forward (MASIC.py:472-506) in one launch.  weights / biases: the four conv3x3 stride-2 layers'
    parameters (maskconv.0, .2, .4, .6).  Returns the (n,3,h/16,w/16) softmax weights (and the NHWC copy)."""
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
    ho, wo = -(-h // 16), -(-w // 16)
    out = torch.empty(n, 3, ho, wo, dtype=torch.float32, device=mask.device)
    out_nhwc = torch.empty(n, ho, wo, 3, dtype=torch.float32, device=mask.device) if nhwc_out else None
    mask2weights_into(mask, ws, bs, out, out_nhwc)
    return (out, out_nhwc) if nhwc_out else out


def softmax_channels(x: torch.Tensor, nhwc_out: bool = False):
    x = _f32c(x)
    n, c, h, w = x.shape
    o1 = torch.empty_like(x)
    o2 = torch.empty(n, h, w, c, dtype=torch.float32, device=x.device) if nhwc_out else None
    softmax_channels_into(x, o1, o2)
    return (o1, o2) if nhwc_out else o1


def nchw_to_nhwc_bf16(x: torch.Tensor, pitch: int, out: Optional[torch.Tensor] = None):
    x = _f32c(x)
    n, c, h, w = x.shape
    if out is None:
        out = torch.empty(n, h, w, pitch, dtype=ACT16, device=x.device)
    nchw_to_nhwc_into(x, out)
    return out


def nhwc_to_nchw_f32(x: torch.Tensor, c: Optional[int] = None, out: Optional[torch.Tensor] = None):
    n, h, w, pitch = x.shape
    c = c or pitch
    if out is None:
        out = torch.empty(n, c, h, w, dtype=torch.float32, device=x.device)
    nhwc_to_nchw_into(x, out)
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
