"""pytorch_msssim.ssim / ms_ssim (version 1.0 semantics, the package the reference's eval loop imports,
coremasic/mywork/test2_real.py:88-114) on the sm_100a MS-SSIM kernel (csrc/msssim.cu)."""
from __future__ import annotations

import torch

from . import torch_ops  # noqa: F401  (registers torch.ops.masic_b200.*)
from .ops import MS_SSIM_WEIGHTS, _need_cuda

__version__ = "1.0.0-masic_b200"


def _check(X, Y, win_size, win_sigma, win):
    if not X.shape == Y.shape:
        raise ValueError(f"Input images should have the same dimensions, but got {X.shape} and {Y.shape}.")
    for d in range(len(X.shape) - 1, 1, -1):           # the package squeezes trailing singleton dimensions
        X = X.squeeze(dim=d)
        Y = Y.squeeze(dim=d)
    if len(X.shape) not in (4, 5):
        raise ValueError(f"Input images should be 4-d or 5-d tensors, but got {X.shape}")
    if win is not None:
        win_size = win.shape[-1]
    if not (win_size % 2 == 1):
        raise ValueError("Window size should be odd.")
    if win is not None or win_size != 11 or win_sigma != 1.5:
        raise NotImplementedError("masic_b200 implements the package's default window: 11 taps, sigma 1.5")
    if len(X.shape) == 5:
        raise NotImplementedError("masic_b200 implements 4-d (N, C, H, W) images only")
    if X.dtype != torch.float32 or Y.dtype != torch.float32:
        raise NotImplementedError(f"masic_b200 implements float32 images only, got {X.dtype} and {Y.dtype}")
    return X, Y


def ssim(X, Y, data_range=255, size_average=True, win_size=11, win_sigma=1.5, win=None, K=(0.01, 0.03),
         nonnegative_ssim=False):
    X, Y = _check(X, Y, win_size, win_sigma, win)
    if min(X.shape[-2:]) < win_size:
        raise NotImplementedError("masic_b200 needs images of at least 11 x 11 (the package skips the filter there)")
    _need_cuda(X, Y)
    v = torch.ops.masic_b200.ms_ssim(X, Y, float(data_range), [1.0], float(K[0]), float(K[1]), bool(nonnegative_ssim))
    return v.mean() if size_average else v.mean(1)


def ms_ssim(X, Y, data_range=255, size_average=True, win_size=11, win_sigma=1.5, win=None, weights=None,
            K=(0.01, 0.03)):
    if not X.shape == Y.shape:
        raise ValueError(f"Input images should have the same dimensions, but got {X.shape} and {Y.shape}.")
    if not X.type() == Y.type():
        raise ValueError(f"Input images should have the same dtype, but got {X.type()} and {Y.type()}.")
    X, Y = _check(X, Y, win_size, win_sigma, win)
    smaller_side = min(X.shape[-2:])
    assert smaller_side > (win_size - 1) * (2 ** 4), \
        "Image size should be larger than %d due to the 4 downsamplings in ms-ssim" % ((win_size - 1) * (2 ** 4))
    weights = list(MS_SSIM_WEIGHTS) if weights is None else [float(w) for w in torch.as_tensor(weights).reshape(-1)]
    if not 1 <= len(weights) <= 5:
        raise NotImplementedError("masic_b200 implements 1 to 5 levels")
    _need_cuda(X, Y)
    v = torch.ops.masic_b200.ms_ssim(X, Y, float(data_range), weights, float(K[0]), float(K[1]), True)
    return v.mean() if size_average else v.mean(1)
