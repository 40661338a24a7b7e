"""Thin Python wrappers of the training-step kernels of the C ABI (include/masic_b200.h, "training" sections).
Each function launches on the current CUDA stream and fails loudly on CPU tensors or a missing library."""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib
from ._lib import check
from .ops import _p, _ptr_array, _s


def lik_grad_scale(num_pixels: int) -> float:
    """d(bpp loss)/d(sum log lik) = -1 / (ln2 * N*H*W)   (newtrain_codec_real.py:73-76)."""
    return -1.0 / (math.log(2.0) * num_pixels)


def gmm_likelihood_train(y, noise, sigma, mu, wl, m, k, scale, *, bound=0.11, lik=None, y_hat_bf=None, y_hat=None,
                         dy=None, dsigma=None, dmu=None, dwl=None):
    npix = y.numel() // m
    check(_lib.load().masic_gmm_likelihood_train(_p(y), _p(noise), _p(sigma), _p(mu), _p(wl), npix, m, k, bound, scale,
                                                 _p(lik), _p(y_hat_bf), 0 if y_hat_bf is None else y_hat_bf.shape[-1],
                                                 _p(y_hat), _p(dy), _p(dsigma), _p(dmu), _p(dwl), _s()),
          "masic_gmm_likelihood_train")


def eb_train(z, noise, n, c, hw, mats, biases, facs, scale, *, z_hat=None, lik=None, zq=None, dz=None, dparams=None):
    check(_lib.load().masic_eb_train(_p(z), _p(noise), n, c, hw, _ptr_array(mats), _ptr_array(biases), _ptr_array(facs),
                                     scale, _p(z_hat), _p(lik), _p(zq), 0 if zq is None else zq.shape[-1], _p(dz),
                                     _p(dparams), _s()), "masic_eb_train")


def eb_aux_loss(quantiles, c, mats, biases, facs, target, loss, dq):
    t = (C.c_float * 3)(*[float(v) for v in target])
    check(_lib.load().masic_eb_aux_loss(_p(quantiles), c, _ptr_array(mats), _ptr_array(biases), _ptr_array(facs), t,
                                        _p(loss), _p(dq), _s()), "masic_eb_aux_loss")


def act_bwd_bias(g, g_coff, c, y, y_coff, act, bias_grad):
    npix = g.numel() // g.shape[-1]
    check(_lib.load().masic_act_bwd_bias(_p(g), g.shape[-1], g_coff, _p(y), 0 if y is None else y.shape[-1], y_coff, act,
                                         npix, c, _p(bias_grad), _s()), "masic_act_bwd_bias")


def gdn_square(x, sq):
    check(_lib.load().masic_gdn_square(_p(x), _p(sq), x.numel(), _s()), "masic_gdn_square")


def gdn_apply(x, norm, inverse, y):
    check(_lib.load().masic_gdn_apply(_p(x), _p(norm), int(inverse), _p(y), x.numel(), _s()), "masic_gdn_apply")


def gdn_bwd_a(g, x, norm, inverse, t, dbeta_prime):
    c = g.shape[-1]
    check(_lib.load().masic_gdn_bwd_a(_p(g), _p(x), _p(norm), int(inverse), _p(t), g.numel() // c, c, _p(dbeta_prime),
                                      _s()), "masic_gdn_bwd_a")


def gdn_bwd_b(u, x, v, dbias):
    c = u.shape[-1]
    check(_lib.load().masic_gdn_bwd_b(_p(u), _p(x), _p(v), u.numel() // c, c, _p(dbias), _s()), "masic_gdn_bwd_b")


class ReparamBatch:
    """Every (dprime, stored, minimum, dstored) reparam backward of a training step as one launch
    (masic_reparam_batch_*); the tensors must stay alive and in place."""

    def __init__(self, jobs):
        import ctypes as C
        lib = _lib.load()
        n = len(jobs)
        self._keep = list(jobs)
        dp = (C.c_void_p * n)(*[j[0].data_ptr() for j in jobs])
        st = (C.c_void_p * n)(*[j[1].data_ptr() for j in jobs])
        ds = (C.c_void_p * n)(*[j[3].data_ptr() for j in jobs])
        ne = (C.c_int * n)(*[j[1].numel() for j in jobs])
        mi = (C.c_float * n)(*[float(j[2]) for j in jobs])
        for j in jobs:
            assert j[0].numel() == j[1].numel() == j[3].numel() and all(t.dtype == torch.float32 and t.is_contiguous() for t in (j[0], j[1], j[3]))
        h = C.c_void_p()
        check(lib.masic_reparam_batch_create(dp, st, ds, ne, mi, None, n, C.byref(h)), "masic_reparam_batch_create")
        self._h, self._lib = h, lib

    def launch(self):
        check(self._lib.masic_reparam_batch_launch(self._h, _s()), "masic_reparam_batch_launch")

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._lib.masic_reparam_batch_destroy(h)
            self._h = None


def reparam_bwd(dprime, stored, minimum, dstored, accumulate=False):
    check(_lib.load().masic_reparam_bwd(_p(dprime), _p(stored), stored.numel(), minimum, int(accumulate), _p(dstored),
                                        _s()), "masic_reparam_bwd")


def latent_prep_train(y, noise, y_abs, y_noisy):
    c = y.shape[-1]
    check(_lib.load().masic_latent_prep_train(_p(y), _p(noise), y.numel() // c, c, _p(y_abs),
                                              0 if y_abs is None else y_abs.shape[-1], _p(y_noisy),
                                              0 if y_noisy is None else y_noisy.shape[-1], _s()),
          "masic_latent_prep_train")


def latent_merge_bwd(y, dy_lik, d_dec, d_ctx, d_abs, dy):
    check(_lib.load().masic_latent_merge_bwd(_p(y), _p(dy_lik), _p(d_dec), _p(d_ctx), _p(d_abs), dy.numel(), _p(dy),
                                             _s()), "masic_latent_merge_bwd")


def add_f32_bf16(a, b, out):
    check(_lib.load().masic_add_f32_bf16(_p(a), _p(b), a.numel(), _p(out), _s()), "masic_add_f32_bf16")


def mask_fuse_fwd(p2, c2t, y1w, noise, mw, fused):
    c2, m = p2.shape[-1], y1w.shape[-1]
    check(_lib.load().masic_mask_fuse_fwd(_p(p2), _p(c2t), c2, _p(y1w), _p(noise), m, _p(mw), y1w.numel() // m,
                                          _p(fused), _s()), "masic_mask_fuse_fwd")


def mask_fuse_bwd(g, p2, c2t, y1w, noise, mw, dp2, dc2, dy1w, dmw):
    c2, m = p2.shape[-1], y1w.shape[-1]
    check(_lib.load().masic_mask_fuse_bwd(_p(g), _p(p2), _p(c2t), c2, _p(y1w), _p(noise), m, _p(mw), y1w.numel() // m,
                                          _p(dp2), _p(dc2), _p(dy1w), _p(dmw), _s()), "masic_mask_fuse_bwd")


def mse_grad(x_hat, x, scale, g, addend=None):
    check(_lib.load().masic_mse_grad(_p(x_hat), _p(x), _p(addend), scale, x.numel(), _p(g), _s()), "masic_mse_grad")


def ms_ssim_buffers(n, c, h, w, device, levels=5):
    """(fwd_scratch, work): device bytes for ms_ssim_fwd and ms_ssim_grad of (n, c, h, w) images (allocate once,
    outside graph capture)."""
    lib = _lib.load()
    fb, wb = lib.masic_ms_ssim_scratch_bytes(n, c, h, w, levels), lib.masic_ms_ssim_bwd_work_bytes(n, c, h, w, levels)
    check(min(int(fb), int(wb), 0), f"masic_ms_ssim_bwd_work_bytes ({levels} levels of {h}x{w} need >= 11x11 each)")
    return (torch.empty(int(fb), dtype=torch.uint8, device=device), torch.empty(int(wb), dtype=torch.uint8, device=device))


def _msssim_args(x_hat, data_range):
    from .ops import MS_SSIM_WEIGHTS
    n, c, h, w = x_hat.shape
    wts = (C.c_float * len(MS_SSIM_WEIGHTS))(*MS_SSIM_WEIGHTS)
    return (n, c, h, w, len(MS_SSIM_WEIGHTS), float(data_range), 0.01, 0.03, wts, 1)


def ms_ssim_fwd(x_hat, x, fwd_scratch, out, data_range=1.0):
    """out (n, c) <- pytorch_msssim.ms_ssim(x_hat, x, data_range, size_average=False) per plane; fwd_scratch keeps
    what ms_ssim_grad reads."""
    check(_lib.load().masic_ms_ssim(_p(x_hat), _p(x), *_msssim_args(x_hat, data_range), _p(fwd_scratch), _p(out), _s()),
          "masic_ms_ssim")


def ms_ssim_grad(x_hat, x, fwd_scratch, scale, g, addend=None, *, work, data_range=1.0):
    """g = scale * d(sum of the per-plane MS-SSIM)/d(x_hat) [+ addend], from the scratch of the ms_ssim_fwd call on
    the same tensors issued before it on the stream."""
    check(_lib.load().masic_ms_ssim_bwd(_p(x_hat), _p(x), *_msssim_args(x_hat, data_range), _p(fwd_scratch), scale,
                                        _p(addend), _p(g), _p(work), _s()), "masic_ms_ssim_bwd")


def warp_bwd(g0, g1, T, dsrc):
    n, c, h, w = dsrc.shape
    check(_lib.load().masic_warp_perspective_bwd(_p(g0), _p(g1), n, c, h, w, g0.shape[2], g0.shape[3], _p(T), _p(dsrc),
                                                 _s()), "masic_warp_perspective_bwd")


def conv_small_bwd(in0, in1, weight, transposed_s1, c_out, ksize, stride, g_out, *, act_out=None, din0=None, din1=None,
                   dweight=None, dbias=None):
    n, c0, h, w = in0.shape
    c1 = 0 if in1 is None else in1.shape[1]
    check(_lib.load().masic_conv_small_bwd(_p(in0), c0, _p(in1), c1, n, h, w, _p(weight), int(transposed_s1), c_out, ksize,
                                           stride, _p(g_out), _p(act_out), _p(din0), _p(din1), _p(dweight), _p(dbias),
                                           _s()), "masic_conv_small_bwd")


def gdn_small_bwd(x, g, beta, gamma, inverse, dx, dbeta_p, dgamma_p, beta_min=1e-6):
    n, c, h, w = x.shape
    check(_lib.load().masic_gdn_small_bwd(_p(x), _p(g), n, c, h * w, _p(beta), _p(gamma), beta_min, int(inverse), _p(dx),
                                          _p(dbeta_p), _p(dgamma_p), _s()), "masic_gdn_small_bwd")


def softmax_channels_bwd(w_nhwc, dw_nhwc, n, c, hw, dlogits):
    check(_lib.load().masic_softmax_channels_bwd(_p(w_nhwc), _p(dw_nhwc), n, c, hw, _p(dlogits), _s()),
          "masic_softmax_channels_bwd")


def wgrad_small(lo, c_lo, hi, dw):
    n, h, w, pitch = lo.shape
    check(_lib.load().masic_wgrad_small(_p(lo), pitch, c_lo, _p(hi), hi.shape[1], n, h, w, _p(dw), _s()),
          "masic_wgrad_small")


def colsum_nchw(g, out):
    n, c = g.shape[0], g.shape[1]
    check(_lib.load().masic_colsum_nchw(_p(g), n, c, g.numel() // (n * c), _p(out), _s()), "masic_colsum_nchw")


def act_bwd_bias_out(g, g_coff, c, y, y_coff, act, dst, dst_coff, bias_grad):
    npix = g.numel() // g.shape[-1]
    check(_lib.load().masic_act_bwd_bias_out(_p(g), g.shape[-1], g_coff, _p(y), 0 if y is None else y.shape[-1], y_coff,
                                             act, npix, c, _p(dst), dst.shape[-1], dst_coff, _p(bias_grad), _s()),
          "masic_act_bwd_bias_out")


def cqe_feature_fuse_bwd(g, self_, other, weights, t_prepared, d_self, d_other, dweights):
    """Backward of masic_cqe_feature_fuse for one view; NHWC buffers, c = the channels of self_ / other."""
    n, h, w, c = self_.shape
    check(_lib.load().masic_cqe_feature_fuse_bwd(_p(g), g.shape[-1], _p(self_), c, _p(other), other.shape[-1], c,
                                                 _p(weights), _p(t_prepared), n, h, w, _p(d_self), d_self.shape[-1],
                                                 _p(d_other), d_other.shape[-1], _p(dweights), _s()),
          "masic_cqe_feature_fuse_bwd")


def cqe_blend_images_bwd(g, a, b, dweights):
    n, _, h, w = a.shape
    check(_lib.load().masic_cqe_blend_images_bwd(_p(g), g.shape[-1], _p(a), _p(b), n, h, w, _p(dweights), _s()),
          "masic_cqe_blend_images_bwd")
