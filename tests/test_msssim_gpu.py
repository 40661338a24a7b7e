"""MS-SSIM on the device (csrc/msssim.cu) against the float64 restatement of pytorch_msssim 1.0 (oracle/msssim.py),
its determinism and batch invariance, the custom op, and PairStream's msssim=True criterion.

Bar: <= 1e-5 absolute per (n, c) value.  Each case prints its measured margins as one JSON line."""
import json
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import msssim as OM

W5 = list(OM.WEIGHTS)
BAR = 1e-5


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from masic_b200 import _lib, torch_ops  # noqa: F401
    _lib.load()
    return torch.device("cuda:0")


def _noisy(shape, dev, seed, sigma=0.05, smooth=True):
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.rand(shape, generator=g, device=dev)
    if smooth:                                   # image-like: spatially correlated content
        x = F.avg_pool2d(F.pad(x, (2, 2, 2, 2), mode="reflect"), 5, stride=1)
        x = (x - x.amin()) / (x.amax() - x.amin())
    y = (x + sigma * torch.randn(shape, generator=g, device=dev)).clamp(0, 1)
    return x.contiguous(), y.contiguous()


def _blurred(shape, dev, seed):
    x, _ = _noisy(shape, dev, seed)
    return x, F.avg_pool2d(F.pad(x, (1, 1, 1, 1), mode="replicate"), 3, stride=1).contiguous()


def _codec_pair(dev, h=192, w=256):
    """A real reconstruction: the engine at g_a_conv4 x 8 (non-degenerate latents), as test_hsic_gpu.py builds it."""
    from masic_b200.hsic import HSIC
    from oracle import hsic as OH
    torch.manual_seed(0)
    net = HSIC().eval()
    with torch.no_grad():
        net.encoder1.g_a_conv4.weight.mul_(8.0)
        net.encoder2.g_a_conv4.weight.mul_(8.0)
    net = net.to(dev)
    g = torch.Generator().manual_seed(100)
    x1, x2 = torch.rand(2, 3, h, w, generator=g), torch.rand(2, 3, h, w, generator=g)
    with torch.no_grad():
        out = net(x1.to(dev), x2.to(dev), OH.synthetic_homography(2, seed=1).to(dev))
    return (torch.cat([out["x1_hat"], out["x2_hat"]]).contiguous(), torch.cat([x1, x2]).to(dev).contiguous())


def _compare(name, x, y, data_range=1.0, weights=None, k=(0.01, 0.03)):
    w = W5 if weights is None else list(weights)
    got_ms = torch.ops.masic_b200.ms_ssim(x, y, data_range, w, k[0], k[1], True).double()
    got_s = torch.ops.masic_b200.ms_ssim(x, y, data_range, [1.0], k[0], k[1], False).double()
    want_ms = OM.ms_ssim_per_channel(x.double(), y.double(), data_range, w, k)
    want_s = OM.ssim_per_channel(x.double(), y.double(), data_range, k)
    e_ms = float((got_ms - want_ms).abs().max())
    e_s = float((got_s - want_s).abs().max())
    print(json.dumps({"case": name, "shape": list(x.shape), "data_range": data_range, "levels": len(w), "K": list(k),
                      "ms_ssim_min": float(want_ms.min()), "ms_ssim_max_abs_err": e_ms,
                      "ssim_min": float(want_s.min()), "ssim_max_abs_err": e_s}))
    assert e_ms <= BAR and e_s <= BAR, (name, e_ms, e_s)
    return got_ms, want_ms


@pytest.mark.parametrize("name,shape,maker,data_range,weights,k", [
    ("noisy_full", (1, 3, 1216, 2176), "noisy", 1.0, None, (0.01, 0.03)),
    ("blurred_full", (1, 3, 1216, 2176), "blurred", 1.0, None, (0.01, 0.03)),
    ("noisy_512_dr255", (1, 3, 512, 512), "noisy", 255.0, None, (0.01, 0.03)),
    ("blurred_512", (1, 3, 512, 512), "blurred", 1.0, None, (0.01, 0.03)),
    ("noisy_321x483_c1", (1, 1, 321, 483), "noisy", 1.0, None, (0.01, 0.03)),
    ("noisy_321x483_c3_weights_K", (1, 3, 321, 483), "noisy", 1.0, (0.1, 0.2, 0.3, 0.25, 0.15), (0.02, 0.05)),
    ("blurred_321x483_dr255_3levels", (1, 3, 321, 483), "blurred", 255.0, (0.3, 0.3, 0.4), (0.01, 0.03)),
    ("noisy_batch4", (4, 3, 200, 232), "noisy", 1.0, None, (0.01, 0.03)),
    ("rough_noise_batch4", (4, 3, 200, 232), "rough", 1.0, None, (0.01, 0.03)),
])
def test_values_against_the_float64_oracle(dev, name, shape, maker, data_range, weights, k):
    if maker == "blurred":
        x, y = _blurred(shape, dev, seed=sum(shape))
    else:
        x, y = _noisy(shape, dev, seed=sum(shape), sigma=0.05 if maker == "noisy" else 0.2, smooth=maker == "noisy")
    _compare(name, x * data_range, y * data_range, data_range, weights, k)


def test_codec_reconstruction_and_size_average(dev):
    from masic_b200 import ops
    xh, x = _codec_pair(dev)
    got, want = _compare("codec_scaled8_192x256", xh, x)
    for sa in (True, False):
        v = ops.ms_ssim(xh, x, data_range=1.0, size_average=sa)
        o = OM.ms_ssim(xh.double(), x.double(), data_range=1.0, size_average=sa)
        assert v.shape == o.shape and float((v.double() - o).abs().max()) <= BAR
        s = ops.ssim(xh * 255, x * 255, size_average=sa, nonnegative_ssim=True)
        o = OM.ssim(xh.double() * 255, x.double() * 255, size_average=sa, nonnegative_ssim=True)
        assert s.shape == o.shape and float((s.double() - o).abs().max()) <= BAR


def test_compat_package_matches_the_oracle(dev):
    from masic_b200.msssim_compat import ms_ssim, ssim
    x, y = _noisy((2, 3, 256, 320), dev, seed=9)
    assert float(ms_ssim(x, y, data_range=1.0)) == pytest.approx(float(OM.ms_ssim(x.double(), y.double(), 1.0)),
                                                                 abs=BAR)
    v = ssim(x * 255, y * 255, size_average=False)
    assert v.shape == (2,)
    assert float((v.double() - OM.ssim(x.double() * 255, y.double() * 255, size_average=False)).abs().max()) <= BAR
    w = torch.tensor([0.5, 0.5])
    assert float(ms_ssim(x, y, data_range=1.0, weights=w)) == pytest.approx(
        float(OM.ms_ssim(x.double(), y.double(), 1.0, weights=[0.5, 0.5])), abs=BAR)


def test_identical_images_give_one(dev):
    for shape in ((1, 3, 1216, 2176), (2, 1, 321, 483)):
        x, _ = _noisy(shape, dev, seed=3)
        ms = torch.ops.masic_b200.ms_ssim(x, x.clone(), 1.0, W5, 0.01, 0.03, True)
        s = torch.ops.masic_b200.ms_ssim(x * 255, x * 255, 255.0, [1.0], 0.01, 0.03, False)
        assert float((ms.double() - 1).abs().max()) <= 1e-7 and float((s.double() - 1).abs().max()) <= 1e-7


def test_inverted_image_takes_the_relu_path(dev):
    """Y = 1 - X: the covariance is negative at every scale, cs < 0, relu -> 0; single-scale SSIM stays negative
    unless nonnegative_ssim."""
    x, _ = _noisy((2, 3, 321, 483), dev, seed=21)
    y = (1.0 - x).contiguous()
    _, cs0 = OM._ssim(x.double(), y.double(), 1.0, OM.gauss_1d())
    assert float(cs0.max()) < 0               # cs of level 0 is negative
    got, want = _compare("inverted_321x483", x, y)
    assert float(want.abs().max()) == 0.0 and float(got.abs().max()) == 0.0
    s = torch.ops.masic_b200.ms_ssim(x, y, 1.0, [1.0], 0.01, 0.03, False)
    s_nn = torch.ops.masic_b200.ms_ssim(x, y, 1.0, [1.0], 0.01, 0.03, True)
    assert float(s.max()) < 0 and float(s_nn.abs().max()) == 0.0


def test_determinism_and_batch_invariance(dev):
    x, y = _noisy((4, 3, 200, 232), dev, seed=4)
    for w, nn in ((W5, True), ([1.0], False)):
        a = torch.ops.masic_b200.ms_ssim(x, y, 1.0, w, 0.01, 0.03, nn)
        b = torch.ops.masic_b200.ms_ssim(x, y, 1.0, w, 0.01, 0.03, nn)
        assert torch.equal(a, b)
        one = torch.cat([torch.ops.masic_b200.ms_ssim(x[i:i + 1].contiguous(), y[i:i + 1].contiguous(), 1.0, w,
                                                      0.01, 0.03, nn) for i in range(4)])
        assert torch.equal(a, one)


def test_custom_op_passes_opcheck(dev):
    x, y = _noisy((2, 3, 176, 200), dev, seed=8)
    torch.library.opcheck(torch.ops.masic_b200.ms_ssim.default, (x, y, 1.0, W5, 0.01, 0.03, True),
                          test_utils=("test_schema", "test_faketensor"))
    torch.library.opcheck(torch.ops.masic_b200.ms_ssim.default, (x, y, 255.0, [1.0], 0.01, 0.03, False),
                          test_utils=("test_schema", "test_faketensor"))


def test_pair_stream_reports_ms_ssim(dev):
    """msssim=True: the 2 x 3 per-channel values read back with the criterion equal the op on outputs() bit for bit;
    bpp, PSNR and the reconstructions do not move; a default submission keeps today's keys."""
    from masic_b200.hsic import HSIC
    torch.manual_seed(0)
    net = HSIC().eval().to(dev)
    h, w = 192, 256
    g = torch.Generator().manual_seed(11)
    x1, x2 = torch.rand(3, 3, h, w, generator=g), torch.rand(3, 3, h, w, generator=g)
    from oracle import hsic as OH
    Hm = OH.synthetic_homography(3, seed=1)
    x1p, x2p, Hp = x1.pin_memory(), x2.pin_memory(), Hm.pin_memory()
    ps = net.pair_stream(h, w, dev, lmbda=0.001)
    base_keys = {"bpp_y1", "bpp_y2", "bpp_z1", "bpp_z2", "mse1", "mse2", "loss"}
    for i in range(3):
        t0 = ps.submit(x1p[i:i + 1], x2p[i:i + 1], Hp[i:i + 1])
        r0 = ps.result(t0)
        rec0 = {k: ps.outputs()[k].clone() for k in ("x1_hat", "x2_hat")}
        assert set(r0[3]) == base_keys
        t1 = ps.submit(x1p[i:i + 1], x2p[i:i + 1], Hp[i:i + 1], msssim=True)
        r1 = ps.result(t1)
        assert r1[:3] == r0[:3] and all(r1[3][k] == r0[3][k] for k in base_keys)
        assert set(r1[3]) == base_keys | {"msssim1", "msssim2", "msssim1_db", "msssim2_db"}
        o = ps.outputs()
        for k in ("x1_hat", "x2_hat"):
            assert torch.equal(o[k], rec0[k])
        per_ch = ps.slots[t1 % ps.depth]["res_h"][8:14]
        for v, (k, x) in enumerate((("x1_hat", x1), ("x2_hat", x2))):
            xd = x[i:i + 1].to(dev)
            op = torch.ops.masic_b200.ms_ssim(o[k], xd, 1.0, W5, 0.01, 0.03, True)
            assert torch.equal(op.cpu().reshape(3), per_ch[3 * v:3 * v + 3]), (op, per_ch)
            want = float(OM.ms_ssim(o[k].double(), xd.double(), data_range=1.0))
            assert r1[3][f"msssim{v + 1}"] == pytest.approx(float(op.mean()), abs=1e-7)
            assert r1[3][f"msssim{v + 1}"] == pytest.approx(want, abs=BAR)
            assert r1[3][f"msssim{v + 1}_db"] == pytest.approx(-10 * math.log10(1 - r1[3][f"msssim{v + 1}"]))
    with pytest.raises(ValueError):
        ps.submit(x1p[0:1], x2p[0:1], Hp[0:1], criterion=False, msssim=True)
