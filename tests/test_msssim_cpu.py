"""MS-SSIM without a GPU: the float64 restatement of pytorch_msssim 1.0 (oracle/msssim.py) against a second,
independent coding of the same definition, the pooling rule at odd sizes, the custom op's registration, the
`pytorch_msssim` compat package's errors, and the C entry points' argument checks."""
import ctypes as C
import math
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
from scipy.ndimage import correlate1d

from masic_b200 import _lib
from masic_b200.build import build
from oracle import msssim as OM

ROOT = Path(__file__).resolve().parents[1]


# ----------------------------------------------------------------------------- independent numpy coding
def _np_filter(x, g):
    """valid correlation with the 1-D window along H and W: the centred 'constant' correlation, cropped"""
    r = len(g) // 2
    out = correlate1d(x, g, axis=2, mode="constant")[:, :, r:x.shape[2] - r]
    return correlate1d(out, g, axis=3, mode="constant")[:, :, :, r:x.shape[3] - r]


def _np_pool(x):
    """2x2 windows over the input zero-padded by (h % 2, w % 2) at the front, every window divided by 4"""
    n, c, h, w = x.shape
    ph, pw = h % 2, w % 2
    ho, wo = (h + 2 * ph) // 2, (w + 2 * pw) // 2
    xp = np.zeros((n, c, 2 * ho, 2 * wo))
    xp[:, :, ph:ph + h, pw:pw + w] = x[:, :, :2 * ho - ph, :2 * wo - pw]
    return xp.reshape(n, c, ho, 2, wo, 2).sum(axis=(3, 5)) / 4.0


def _np_levels(x, y, g, data_range, k, levels):
    c1, c2 = (k[0] * data_range) ** 2, (k[1] * data_range) ** 2
    out = []
    for lv in range(levels):
        if lv:
            x, y = _np_pool(x), _np_pool(y)
        mx, my = _np_filter(x, g), _np_filter(y, g)
        vx, vy, vxy = _np_filter(x * x, g) - mx * mx, _np_filter(y * y, g) - my * my, _np_filter(x * y, g) - mx * my
        cs = (2 * vxy + c2) / (vx + vy + c2)
        ss = (2 * mx * my + c1) / (mx * mx + my * my + c1) * cs
        out.append((ss.mean(axis=(2, 3)), cs.mean(axis=(2, 3))))
    return out


def _np_ms_ssim(x, y, g, data_range, weights, k):
    lv = _np_levels(x, y, g, data_range, k, len(weights))
    v = np.ones(x.shape[:2])
    for i, (ss, cs) in enumerate(lv):
        v = v * np.maximum(cs if i < len(weights) - 1 else ss, 0.0) ** weights[i]
    return v


def _pair(shape, seed):
    rng = np.random.default_rng(seed)
    x = rng.random(shape)
    y = np.clip(x + 0.1 * rng.standard_normal(shape), 0.0, 1.0)
    return x, y


def test_window_taps_are_the_float32_gaussian():
    g = OM.gauss_1d()[0, 0]
    assert g.dtype == torch.float32 and g.shape == (11,)
    d = np.arange(11) - 5.0
    e = np.exp(-d * d / (2 * 1.5 ** 2))
    assert np.abs(g.double().numpy() - e / e.sum()).max() <= 1e-7
    assert abs(float(g.double().sum()) - 1.0) <= 1e-6


@pytest.mark.parametrize("shape", [(2, 3, 176, 192), (1, 2, 161, 183), (1, 1, 170, 165)])
@pytest.mark.parametrize("data_range,weights,k", [(1.0, None, (0.01, 0.03)), (255.0, (0.2, 0.3, 0.5), (0.02, 0.05))])
def test_oracle_matches_an_independent_numpy_coding(shape, data_range, weights, k):
    x, y = _pair(shape, seed=sum(shape))
    x, y = x * data_range, y * data_range
    g = OM.gauss_1d()[0, 0].double().numpy()
    w = OM.WEIGHTS if weights is None else weights
    want = _np_ms_ssim(x, y, g, data_range, w, k)
    got = OM.ms_ssim_per_channel(torch.from_numpy(x), torch.from_numpy(y), data_range, weights, k).numpy()
    assert np.abs(got - want).max() <= 1e-12, (got, want)
    ss0 = _np_levels(x, y, g, data_range, k, 1)[0][0]
    got_s = OM.ssim_per_channel(torch.from_numpy(x), torch.from_numpy(y), data_range, k).numpy()
    assert np.abs(got_s - ss0).max() <= 1e-12
    assert OM.ms_ssim(torch.from_numpy(x), torch.from_numpy(y), data_range, False, weights, k).shape == (shape[0],)


def test_oracle_of_identical_images_is_one():
    x, _ = _pair((2, 3, 180, 200), seed=5)
    t = torch.from_numpy(x)
    assert float(OM.ms_ssim(t, t, data_range=1.0)) == pytest.approx(1.0, abs=1e-14)
    assert float(OM.ssim(t, t, data_range=1.0)) == pytest.approx(1.0, abs=1e-14)


def test_pooling_pitfall_at_odd_sizes():
    x = torch.arange(25, dtype=torch.float64).view(1, 1, 5, 5)
    p = OM.pool(x)
    assert p.shape == (1, 1, 3, 3)
    assert p[0, 0, 0].tolist() == [0.0, 0.75, 1.75]
    assert np.array_equal(p.numpy(), _np_pool(x.numpy()))
    sizes = [(321, 483)]
    for _ in range(4):
        sizes.append(tuple(OM.pool(torch.zeros(1, 1, *sizes[-1])).shape[2:]))
    assert [s[0] for s in sizes] == [321, 161, 81, 41, 21] and [s[1] for s in sizes] == [483, 242, 121, 61, 31]


def test_custom_op_is_registered_with_a_fake_impl():
    from masic_b200 import torch_ops
    assert "ms_ssim" in torch_ops.OPS
    assert torch.ops.masic_b200.ms_ssim.default._schema.name == "masic_b200::ms_ssim"
    m = torch.empty(4, 3, 200, 232, device="meta")
    out = torch.ops.masic_b200.ms_ssim(m, m, 1.0, list(OM.WEIGHTS), 0.01, 0.03, True)
    assert out.shape == (4, 3) and out.dtype == torch.float32
    with pytest.raises((NotImplementedError, RuntimeError)):
        torch.ops.masic_b200.ms_ssim(torch.zeros(1, 1, 32, 32), torch.zeros(1, 1, 32, 32), 1.0, [1.0], 0.01, 0.03, False)
    from masic_b200 import ops
    with pytest.raises(_lib.MasicError):
        ops.ms_ssim(torch.zeros(1, 3, 200, 200), torch.zeros(1, 3, 200, 200))
    with pytest.raises(_lib.MasicError):
        ops.ssim(torch.zeros(1, 3, 64, 64), torch.zeros(1, 3, 64, 64))


_COMPAT = r"""
import sys, torch
sys.path[:0] = [%(root)r, %(root)r + '/masic_b200/compat']
import pytorch_msssim
from pytorch_msssim import ms_ssim, ssim
assert '/masic_b200/compat/' in pytorch_msssim.__file__
def raises(exc, fn, *a, **k):
    try:
        fn(*a, **k)
    except exc as e:
        return str(e)
    raise SystemExit(f'{fn.__name__}{k} did not raise {exc.__name__}')
x = torch.zeros(1, 3, 200, 200)
assert 'same dimensions' in raises(ValueError, ms_ssim, x, torch.zeros(1, 3, 200, 201))
assert 'same dimensions' in raises(ValueError, ssim, x, torch.zeros(1, 1, 200, 200))
assert 'same dtype' in raises(ValueError, ms_ssim, x, x.double())
assert '4-d or 5-d' in raises(ValueError, ssim, torch.zeros(3, 200, 200), torch.zeros(3, 200, 200))
assert 'odd' in raises(ValueError, ms_ssim, x, x, win_size=10)
assert 'larger than 160' in raises(AssertionError, ms_ssim, torch.zeros(1, 3, 160, 300), torch.zeros(1, 3, 160, 300))
raises(NotImplementedError, ms_ssim, x, x, win_size=7)
raises(NotImplementedError, ssim, x, x, win_sigma=2.0)
raises(NotImplementedError, ssim, x, x, win=torch.ones(1, 1, 11) / 11)
raises(NotImplementedError, ms_ssim, torch.zeros(1, 3, 8, 200, 200), torch.zeros(1, 3, 8, 200, 200))
raises(NotImplementedError, ms_ssim, x.double(), x.double())
raises(NotImplementedError, ssim, x.half(), x.half())
from masic_b200._lib import MasicError
raises(MasicError, ms_ssim, x, x)                       # CPU tensors: no fallback
print('OK')
"""


def test_compat_package_imports_and_raises_the_documented_errors():
    out = subprocess.run([sys.executable, "-c", _COMPAT % {"root": str(ROOT)}], capture_output=True, text=True,
                         timeout=300)
    assert out.returncode == 0 and out.stdout.strip().endswith("OK"), out.stdout[-2000:] + out.stderr[-3000:]


def test_entry_points_reject_bad_arguments_without_a_gpu():
    build()
    lib = _lib.load()
    EINVAL = -1
    assert lib.masic_ms_ssim_scratch_bytes(1, 3, 1216, 2176, 5) > 0
    assert lib.masic_ms_ssim_scratch_bytes(1, 3, 161, 161, 5) > 0          # 161 -> 81 -> 41 -> 21 -> 11
    for args in ((0, 3, 256, 256, 5), (1, -1, 256, 256, 5), (1, 3, 0, 256, 5), (1, 3, 256, 256, 0),
                 (1, 3, 256, 256, 6), (1, 3, 160, 256, 5), (1, 3, 10, 10, 1), (1, 1, 100, 20, 2)):
        assert lib.masic_ms_ssim_scratch_bytes(*args) == EINVAL, args
    w = (C.c_float * 5)(*OM.WEIGHTS)
    p = C.c_void_p(256)                          # never dereferenced: every call below is rejected first
    good = dict(x=p, y=p, n=1, c=3, h=256, w=256, levels=5, dr=1.0, k1=0.01, k2=0.03, wt=w, nn=1, scratch=p, out=p)

    def call(**kw):
        a = {**good, **kw}
        return lib.masic_ms_ssim(a["x"], a["y"], a["n"], a["c"], a["h"], a["w"], a["levels"], a["dr"], a["k1"],
                                 a["k2"], a["wt"], a["nn"], a["scratch"], a["out"], None)
    for kw in (dict(x=None), dict(y=None), dict(wt=None), dict(scratch=None), dict(out=None), dict(n=0), dict(c=0),
               dict(h=-5), dict(w=0), dict(levels=0), dict(levels=6), dict(h=150), dict(w=160, levels=5),
               dict(h=10, levels=1), dict(dr=0.0), dict(dr=math.nan), dict(k1=-0.01)):
        assert call(**kw) == EINVAL, kw
