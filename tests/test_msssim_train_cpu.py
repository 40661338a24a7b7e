"""Training for MS-SSIM without a GPU: the float64 autograd gradient of oracle/msssim.py (the reference the CUDA
backward is tested against) checked by central finite differences, including a plane whose relu clamps, and the
argument checks of masic_ms_ssim_bwd and of the trainer's `metric` option."""
import ctypes as C

import pytest
import torch

from masic_b200 import _lib
from masic_b200.build import build
from oracle import msssim as OM


def _pair(n, c, h, w, seed, noise=0.03):
    g = torch.Generator().manual_seed(seed)
    base = torch.rand(n, c, h // 8 + 2, w // 8 + 2, generator=g, dtype=torch.float64)
    x = torch.nn.functional.interpolate(base, size=(h, w), mode="bilinear", align_corners=False)
    x_hat = (x + noise * torch.randn(n, c, h, w, generator=g, dtype=torch.float64)).clamp(0.0, 1.0)
    return x_hat, x


def _total(x_hat, x):
    return OM.ms_ssim_per_channel(x_hat, x, data_range=1.0).sum()


def _autograd(x_hat, x):
    xr = x_hat.clone().requires_grad_()
    v = _total(xr, x)
    v.backward()
    return v.detach(), xr.grad


def _central_differences(x_hat, x, idx, eps=1e-5):
    out = []
    for i in idx:
        xp, xm = x_hat.clone(), x_hat.clone()
        xp.view(-1)[i] += eps
        xm.view(-1)[i] -= eps
        out.append(float(_total(xp, x) - _total(xm, x)) / (2 * eps))
    return torch.tensor(out, dtype=torch.float64)


def test_reference_gradient_matches_finite_differences():
    # 161 x 177: the pyramid is 161x177, 81x89, 41x45, 21x23, 11x12, odd (padded pooling) at almost every level
    x_hat, x = _pair(1, 2, 161, 177, 1)
    _, grad = _autograd(x_hat, x)
    g = torch.Generator().manual_seed(2)
    idx = torch.randint(0, x_hat.numel(), (20,), generator=g).tolist()
    idx[0] = 0                                         # a corner pixel, inside the first pooling window's pad
    fd = _central_differences(x_hat, x, idx)
    want = grad.view(-1)[idx]
    assert torch.all(want != 0)
    # the differences round at ~1e-16 / eps of the value: about 1e-11 here, against gradients of ~1e-5
    assert float((fd - want).abs().max()) <= 1e-4 * float(want.abs().max())
    assert float((fd - want).norm() / want.norm()) <= 1e-4


def test_reference_gradient_is_zero_where_relu_clamps():
    # an inverted image: every level's mean cs is negative, relu clamps, the value and the gradient are 0, not NaN
    x_hat, x = _pair(1, 1, 161, 177, 3)
    value, grad = _autograd(1.0 - x, x)
    assert float(value) == 0.0
    assert torch.isfinite(grad).all() and float(grad.abs().max()) == 0.0
    fd = _central_differences(1.0 - x, x, [5, 1000, 20000])
    assert float(fd.abs().max()) == 0.0
    # one clamped plane next to a normal one: the normal plane's gradient is untouched
    both = torch.cat([x_hat, 1.0 - x], dim=1)
    _, g2 = _autograd(both, x.repeat(1, 2, 1, 1))
    _, g1 = _autograd(x_hat, x)
    assert torch.equal(g2[:, :1], g1) and float(g2[:, 1:].abs().max()) == 0.0


@pytest.fixture(scope="module")
def lib():
    build()
    return _lib.load()


def test_bwd_entry_points_reject_bad_arguments(lib):
    assert lib.masic_ms_ssim_bwd_work_bytes(2, 3, 512, 896, 5) > 0
    assert lib.masic_ms_ssim_bwd_work_bytes(1, 3, 161, 177, 5) > 0
    for args in [(0, 3, 256, 256, 5), (1, 0, 256, 256, 5), (1, 3, 160, 256, 5), (1, 3, 256, 10, 1),
                 (1, 3, 256, 256, 0), (1, 3, 256, 256, 6), (1, 3, -1, 256, 5)]:
        assert lib.masic_ms_ssim_bwd_work_bytes(*args) == -1, args
    wts = (C.c_float * 5)(*OM.WEIGHTS)
    p = C.c_void_p(16)                                 # never dereferenced: every call below fails its checks first

    def call(x=p, y=p, n=1, c=3, h=256, w=256, levels=5, dr=1.0, wt=wts, scratch=p, dx=p, work=p):
        return lib.masic_ms_ssim_bwd(x, y, n, c, h, w, levels, dr, 0.01, 0.03, wt, 1, scratch, -1.0, None, dx, work,
                                     None)
    assert call(x=None) == -1
    assert call(y=None) == -1
    assert call(wt=None) == -1
    assert call(scratch=None) == -1
    assert call(dx=None) == -1
    assert call(work=None) == -1
    assert call(dr=0.0) == -1
    assert call(h=160) == -1
    assert call(levels=0) == -1 and call(levels=6) == -1
    assert call(n=0) == -1


def test_trainer_metric_is_checked_before_any_cuda_work():
    from masic_b200.hsic import HSIC
    net = HSIC()
    with pytest.raises(ValueError, match="metric"):
        net.trainer(1, 192, 256, "cpu", metric="ssim")
    with pytest.raises(ValueError, match="160"):
        net.trainer(1, 128, 256, "cpu", metric="ms-ssim")
