"""pytorch_msssim 1.0 (`ssim`, `ms_ssim`), the MS-SSIM the reference's eval loop reports
(coremasic/mywork/test2_real.py:88-114, test3_real.py), restated op for op.

The package is not vendored by the reference and is not installed here, so, as for kornia, this restatement is the
specification.  It computes in the dtype of its inputs: the tests call it on float64 tensors; on float32 CUDA tensors it
is the op sequence the package itself runs (grouped conv2d passes, avg_pool2d, elementwise maps).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)


def gauss_1d(size: int = 11, sigma: float = 1.5) -> torch.Tensor:
    """_fspecial_gauss_1d: float32 taps normalised to sum 1, shape (1, 1, size)."""
    coords = torch.arange(size, dtype=torch.float)
    coords -= size // 2
    g = torch.exp(-(coords ** 2) / (2 * sigma ** 2))
    g /= g.sum()
    return g.unsqueeze(0).unsqueeze(0)


def gaussian_filter(x: torch.Tensor, win: torch.Tensor) -> torch.Tensor:
    """Separable valid correlation per channel (groups = C): along H, then along W."""
    c = x.shape[1]
    w = win.to(x.device, x.dtype).repeat(c, 1, 1).unsqueeze(1)      # (C, 1, 1, size)
    out = F.conv2d(x, w.transpose(2, 3), groups=c)
    return F.conv2d(out, w, groups=c)


def _ssim(X, Y, data_range, win, K=(0.01, 0.03)):
    """(ssim_per_channel, cs), each (N, C)."""
    K1, K2 = K
    C1 = (K1 * data_range) ** 2
    C2 = (K2 * data_range) ** 2
    mu1 = gaussian_filter(X, win)
    mu2 = gaussian_filter(Y, win)
    mu1_sq, mu2_sq, mu1_mu2 = mu1.pow(2), mu2.pow(2), mu1 * mu2
    sigma1_sq = gaussian_filter(X * X, win) - mu1_sq
    sigma2_sq = gaussian_filter(Y * Y, win) - mu2_sq
    sigma12 = gaussian_filter(X * Y, win) - mu1_mu2
    cs_map = (2 * sigma12 + C2) / (sigma1_sq + sigma2_sq + C2)
    ssim_map = ((2 * mu1_mu2 + C1) / (mu1_sq + mu2_sq + C1)) * cs_map
    return torch.flatten(ssim_map, 2).mean(-1), torch.flatten(cs_map, 2).mean(-1)


def pool(x: torch.Tensor) -> torch.Tensor:
    """The pyramid step: avg_pool2d(2, padding (h % 2, w % 2)), count_include_pad=True.  At an odd size the first
    window holds one zero pad and still divides by 4."""
    return F.avg_pool2d(x, kernel_size=2, padding=[s % 2 for s in x.shape[2:]])


def ssim_per_channel(X, Y, data_range=255, K=(0.01, 0.03), nonnegative_ssim=False):
    s, _ = _ssim(X, Y, data_range, gauss_1d(), K)
    return torch.relu(s) if nonnegative_ssim else s


def ms_ssim_per_channel(X, Y, data_range=255, weights=None, K=(0.01, 0.03)):
    """(N, C): prod over levels of relu(cs_l) ** w_l, the last level's relu(ssim) ** w_L instead of its cs."""
    assert min(X.shape[-2:]) > 10 * 2 ** 4, "Image size should be larger than 160 due to the 4 downsamplings in ms-ssim"
    weights = X.new_tensor(WEIGHTS if weights is None else weights)
    win = gauss_1d()
    mcs = []
    for i in range(weights.shape[0]):
        s, cs = _ssim(X, Y, data_range, win, K)
        if i < weights.shape[0] - 1:
            mcs.append(torch.relu(cs))
            X, Y = pool(X), pool(Y)
    vals = torch.stack(mcs + [torch.relu(s)], dim=0)
    return torch.prod(vals ** weights.view(-1, 1, 1), dim=0)


def ms_ssim(X, Y, data_range=255, size_average=True, weights=None, K=(0.01, 0.03)):
    v = ms_ssim_per_channel(X, Y, data_range, weights, K)
    return v.mean() if size_average else v.mean(1)


def ssim(X, Y, data_range=255, size_average=True, K=(0.01, 0.03), nonnegative_ssim=False):
    v = ssim_per_channel(X, Y, data_range, K, nonnegative_ssim)
    return v.mean() if size_average else v.mean(1)
