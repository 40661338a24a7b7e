"""Pairs of any size on the B200: the pad and homography kernels, and every entry point of the codec at sizes that are
not multiples of 64, checked against the definition (masic_b200/padding.py): run the 64-multiple path on the
zero-padded pair with the homography T H T^-1, crop the images back, divide bpp by the original pixel count."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

VIEWS = ("x1_hat", "x2_hat")
CROPPED = ("x1_hat", "x2_hat", "x1_mask_R", "x1_mask_L")


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from masic_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def codec(dev):
    """Seeded HSIC with g_a_conv4 x 8, so that the latents are far from all-zero (bitmaps and payloads are non-trivial)."""
    from masic_b200.hsic import HSIC
    torch.manual_seed(0)
    net = HSIC().eval()
    with torch.no_grad():
        net.encoder1.g_a_conv4.weight.mul_(8.0)
        net.encoder2.g_a_conv4.weight.mul_(8.0)
    net = net.to(dev)
    net.update(force=True)
    return net


def _pairs(n, h, w, seed, u8=False):
    from oracle import hsic as OH
    g = torch.Generator().manual_seed(seed)
    if u8:
        x1 = torch.randint(0, 256, (n, 3, h, w), generator=g, dtype=torch.uint8)
        x2 = torch.randint(0, 256, (n, 3, h, w), generator=g, dtype=torch.uint8)
    else:
        x1, x2 = torch.rand(n, 3, h, w, generator=g), torch.rand(n, 3, h, w, generator=g)
    return x1, x2, OH.synthetic_homography(n, seed=seed + 1)


def _h_padded(Hm: torch.Tensor, pad) -> torch.Tensor:
    """T H T^-1 in float64, each product and sum in the order the kernel rounds them, rounded once to float32."""
    m = Hm.detach().cpu().double().numpy().reshape(-1, 3, 3)
    t, l = float(pad.top), float(pad.left)
    out = np.empty_like(m)
    c = (m[:, :, 2] - l * m[:, :, 0]) - t * m[:, :, 1]          # column 2 of H T^-1
    out[:, 0, :2] = m[:, 0, :2] + l * m[:, 2, :2]
    out[:, 1, :2] = m[:, 1, :2] + t * m[:, 2, :2]
    out[:, 0, 2] = c[:, 0] + l * c[:, 2]
    out[:, 1, 2] = c[:, 1] + t * c[:, 2]
    out[:, 2, :2] = m[:, 2, :2]
    out[:, 2, 2] = c[:, 2]
    return torch.from_numpy(out.astype(np.float32)).reshape(Hm.shape)


def _defined(codec, x1, x2, Hm, pad):
    """The definition: HSIC.forward of the padded pair, images cropped back."""
    with torch.no_grad():
        out = codec(F.pad(x1, pad.pad_args()), F.pad(x2, pad.pad_args()), _h_padded(Hm, pad).to(x1.device))
    return {**out, **{k: pad.crop(out[k]).contiguous() for k in CROPPED}}


# ------------------------------------------------------------------------------------------------------------ kernels
def test_pad_image_is_f_pad(dev):
    """Both outputs for uint8 (ToTensor) and float32 sources, n = 2, several sizes; each padded buffer is reused by a
    pair of another size first (and starts as NaN), so every element, border included, must be written."""
    from masic_b200 import _lib, ops
    from masic_b200.padding import padding_for
    g = torch.Generator().manual_seed(1)
    groups = [[(375, 1242), (380, 1250)], [(200, 333), (250, 380)], [(100, 130), (65, 129)], [(1, 1), (63, 63)]]
    for sizes in groups:
        pads = [padding_for(*s) for s in sizes]
        assert len({(p.hp, p.wp) for p in pads}) == 1
        for u8 in (True, False):
            dst = torch.full((2, 3, pads[0].hp, pads[0].wp), float("nan"), device=dev)
            for pad in pads:
                x = (torch.randint(0, 256, (2, 3, pad.h, pad.w), generator=g, dtype=torch.uint8) if u8
                     else torch.rand(2, 3, pad.h, pad.w, generator=g))
                unit = x.float().div(255) if u8 else x                 # ToTensor on the host
                unpadded = torch.full((2, 3, pad.h, pad.w), float("nan"), device=dev)
                pad.image_into(x.to(dev), dst, unpadded=unpadded)
                assert torch.equal(dst.cpu(), F.pad(unit, pad.pad_args())), (pad, u8)
                assert torch.equal(unpadded.cpu(), unit)
                pad.image_into(x.to(dev), dst)                          # without the second output
                assert torch.equal(dst.cpu(), F.pad(unit, pad.pad_args()))
                if u8:                                                  # the same bits as masic_u8_to_unit_f32
                    xd, ref = x.to(dev), torch.empty_like(unpadded)
                    _lib.check(_lib.load().masic_u8_to_unit_f32(xd.data_ptr(), xd.numel(), ref.data_ptr(),
                                                               torch.cuda.current_stream().cuda_stream), "u8")
                    assert torch.equal(unpadded, ref)
    # a frame whose width is not a multiple of 4 takes the scalar stores
    x = torch.rand(1, 2, 5, 7, generator=g)
    dst = torch.full((1, 2, 9, 10), float("nan"), device=dev)
    ops.pad_image_into(x.to(dev), dst, 3, 2)
    assert torch.equal(dst.cpu(), F.pad(x, (2, 1, 3, 1)))


def test_homography_pad_kernel(dev):
    """Bit-identical to the host float64 expression in the kernel's order, within 1 fp32 ulp of T H T^-1 by matrix
    products in float64, and in place."""
    from masic_b200.padding import padding_for
    from oracle import hsic as OH
    Hm = OH.synthetic_homography(64, seed=9)
    Hm[::3] *= torch.rand(22, 1, 1, generator=torch.Generator().manual_seed(2)) * 3 + 0.1     # unnormalised too
    for h, w in ((375, 1242), (200, 333), (1, 1), (1216, 2176), (860, 1080)):
        pad = padding_for(h, w)
        out = torch.full((64, 3, 3), float("nan"), device=dev)
        hd = Hm.to(dev).contiguous()
        pad.homography_into(hd, out)
        assert torch.equal(out.cpu(), _h_padded(Hm, pad))
        T = torch.tensor([[1, 0, pad.left], [0, 1, pad.top], [0, 0, 1]], dtype=torch.float64)
        ref = (T @ Hm.double() @ torch.linalg.inv(T)).float()
        assert (out.cpu().view(torch.int32) - ref.view(torch.int32)).abs().max() <= 1
        pad.homography_into(hd, hd)
        assert torch.equal(hd, out)


# ------------------------------------------------------------------------------------------------------------ forward
@pytest.mark.parametrize("hw", [(375, 1242), (200, 333), (100, 130)], ids=lambda s: f"{s[0]}x{s[1]}")
@pytest.mark.parametrize("batch", [1, 2])
def test_forward_is_the_defined_composition(dev, codec, hw, batch):
    from masic_b200.padding import padding_for
    pad = padding_for(*hw)
    x1, x2, Hm = _pairs(batch, *hw, seed=3 + batch)
    x1, x2, Hm = x1.to(dev), x2.to(dev), Hm.to(dev)
    want = _defined(codec, x1, x2, Hm, pad)
    with torch.no_grad():
        got = codec(x1, x2, Hm)
    for k in CROPPED:
        assert got[k].shape[-2:] == hw and torch.equal(got[k], want[k]), k
    for k in ("y1_hat", "z1_hat"):
        assert got[k].shape[-2:] == want[k].shape[-2:] == (pad.hp // (16 if k[0] == "y" else 64),
                                                          pad.wp // (16 if k[0] == "y" else 64))
        assert torch.equal(got[k], want[k]), k
    for k in want["likelihoods"]:
        assert torch.equal(got["likelihoods"][k], want["likelihoods"][k]), k
    with torch.no_grad():                                    # clone=False hands out the staging buffers
        again = codec(x1, x2, Hm, clone=False)
    assert torch.equal(again["x1_hat"], want["x1_hat"])


def test_forward_at_a_multiple_of_64_is_todays_call(dev, codec):
    x1, x2, Hm = _pairs(1, 384, 1280, seed=8)
    x1, x2, Hm = x1.to(dev), x2.to(dev), Hm.to(dev)
    with torch.no_grad():
        got = codec(x1, x2, Hm)
        o = codec.engine_for(1, 384, 1280, dev).run(x1, x2, Hm)
        for k in CROPPED + ("y1_hat", "z1_hat"):
            assert torch.equal(got[k], o[k]), k


# ------------------------------------------------------------------------------------------------------------ stream
def _enhancer(dev):
    from masic_b200.cqe import Independent_EN
    torch.manual_seed(3)
    en = Independent_EN().eval()
    with torch.no_grad():
        en.conv2.weight.mul_(0.03)
        en.conv2.bias.mul_(0.03)
    return en.to(dev)


def _lpips(dev):
    from masic_b200.lpips import LPIPS
    from oracle import lpips as OL
    net = LPIPS(pretrained=False, pnet_rand=True, verbose=False)
    net.load_state_dict(OL.random_state_dict(3))
    return net.to(dev)


@pytest.mark.parametrize("u8", [False, True], ids=["float32", "uint8"])
@pytest.mark.parametrize("depth", [2, 3])
def test_pair_stream_at_375x1242(dev, codec, depth, u8):
    """Pairs in flight (results read one pair behind): every number, reconstruction and enhanced pair equals the public
    two-step path: cropped forward, then bpp_and_psnr / ops.ms_ssim / LPIPS / Independent_EN.forward(crop, h)."""
    from masic_b200 import ops
    from masic_b200.hsic import bpp_and_psnr
    h, w, n, lmbda = 375, 1242, 3, 0.001
    en, lp = _enhancer(dev), _lpips(dev)
    x1, x2, Hm = _pairs(n, h, w, seed=20 + depth, u8=u8)
    ps = codec.pair_stream(h, w, dev, depth=depth, lmbda=lmbda)
    ps.attach_enhancement(en)
    ps.attach_lpips(lp)
    x1p, x2p, Hp = x1.pin_memory(), x2.pin_memory(), Hm.pin_memory()
    tickets = []

    def check(i, t, enhance):
        r = ps.result(t)
        rec = ps.reconstructions(t)
        xs = [(x[i:i + 1].float().div(255) if u8 else x[i:i + 1]).to(dev) for x in (x1, x2)]
        hd = Hm[i:i + 1].to(dev)
        with torch.no_grad():
            out = codec(xs[0], xs[1], hd)
            enh = en(out["x1_hat"], out["x2_hat"], hd) if enhance else out
        # the public criterion, evaluated in float64 so that its own float32 rounding does not enter the comparison
        out64 = {"likelihoods": {k: v.double() for k, v in out["likelihoods"].items()},
                 **{k: out[k].double() for k in VIEWS}}
        bpp, p1, p2 = bpp_and_psnr(out64, *(x.double() for x in xs))
        assert r[0] == pytest.approx(float(bpp), rel=2e-6)
        for v, k in enumerate(VIEWS):
            assert torch.equal(rec[v], enh[k].cpu()), (i, k)
            mse = float(((enh[k].double() - xs[v].double()) ** 2).mean())
            assert r[3][f"mse{v + 1}"] == pytest.approx(mse, rel=2e-6)
            assert r[1 + v] == pytest.approx(10 * math.log10(1 / mse), abs=1e-4)
            assert r[3][f"msssim{v + 1}"] == pytest.approx(float(ops.ms_ssim(enh[k], xs[v], data_range=1.0)), abs=1e-7)
            assert r[3][f"lpips{v + 1}"] == float(lp(enh[k], xs[v], normalize=True))
        if enhance:
            assert r[3]["codec_psnr1"] == pytest.approx(float(p1), abs=1e-4)
            assert r[3]["codec_psnr2"] == pytest.approx(float(p2), abs=1e-4)
        return out, enh

    for i in range(n):
        enhance = i != 1
        tickets.append(ps.submit(x1p[i:i + 1], x2p[i:i + 1], Hp[i:i + 1], want_recon=True, msssim=True, lpips=True,
                                 enhance=enhance))
        if i >= 1:
            check(i - 1, tickets[i - 1], i - 1 != 1)
    out, enh = check(n - 1, tickets[-1], True)
    for k in VIEWS:
        assert torch.equal(ps.enhanced_outputs()[k], enh[k])
        assert torch.equal(ps.outputs()[k], out[k])
    for k in ("x1_mask_R", "x1_mask_L", "y1_hat", "lik_y1"):
        want = out[k] if k in out else out["likelihoods"]["y1"]
        assert torch.equal(ps.outputs()[k], want), k


def test_pair_stream_patches_at_an_odd_size(dev, codec):
    """submit_patches equals submit with Net.homography(..., img_hw=(h, w)) of the original size."""
    from masic_b200.udh import Net
    from oracle import udh as OU
    h, w = 375, 1242
    torch.manual_seed(1)
    udh = Net().eval()
    with torch.no_grad():
        udh.fc[5].weight.mul_(200.0)
    udh = udh.to(dev)
    x1, x2, _ = _pairs(1, h, w, seed=31, u8=True)
    a, b, corners = OU.synthetic_patches(1, seed=2)
    with torch.no_grad():
        hm = udh.homography(a.to(dev), b.to(dev), corners.to(dev), img_hw=(h, w))
    ps = codec.pair_stream(h, w, dev, depth=2)
    ps.attach_homography_net(udh)
    x1p, x2p = x1.pin_memory(), x2.pin_memory()
    tp = ps.submit_patches(x1p, x2p, a.pin_memory(), b.pin_memory(), corners.pin_memory(), want_recon=True)
    rp = ps.result(tp)
    rec_p = [t.clone() for t in ps.reconstructions(tp)]
    ts = ps.submit(x1p, x2p, hm.cpu().pin_memory(), want_recon=True)
    assert rp == ps.result(ts)
    for a_, b_ in zip(rec_p, ps.reconstructions(ts)):
        assert torch.equal(a_, b_)


# ------------------------------------------------------------------------------------------------------------ bitstreams
@pytest.mark.parametrize("hw,y_order", [((375, 1242), "wavefront_streams"), ((70, 100), "raster"),
                                         ((70, 100), "wavefront"), ((100, 130), "wavefront_streams")],
                         ids=["375x1242-streams", "70x100-raster", "70x100-wavefront", "100x130-streams"])
def test_compress_decompress_at_an_odd_size(dev, codec, tmp_path, hw, y_order):
    from masic_b200.bitstream import _parse_header
    from masic_b200.padding import padding_for
    pad = padding_for(*hw)
    x1, x2, Hm = _pairs(1, *hw, seed=40)
    x1, x2, Hm = x1.to(dev), x2.to(dev), Hm.to(dev)
    want = _defined(codec, x1, x2, Hm, pad)
    with torch.no_grad():
        enc = codec.compress(x1, x2, Hm, "p", str(tmp_path), y_order=y_order)
        dec = codec.decompress(x1, x2, Hm, "p", str(tmp_path), device=dev)
    head = (tmp_path / "p.npz").read_bytes()
    assert _parse_header(head, codec.M)[:2] == hw
    n_bytes = len(head) + (tmp_path / "p.bin").stat().st_size
    assert enc["bpp_real"] == n_bytes * 8 / (2 * hw[0] * hw[1])
    assert torch.equal(enc["y1_hat"], want["y1_hat"])
    for k in VIEWS:
        assert dec[k].shape[-2:] == hw and torch.equal(dec[k], want[k]), k
    assert torch.equal(dec["y1_hat"], want["y1_hat"])


def test_batch_coding_at_an_odd_size(dev, codec, tmp_path):
    """compress_batch / decompress_batch at 200x333, B = 3: byte- and bit-identical to the per-pair API."""
    from masic_b200.padding import padding_for
    h, w, B = 200, 333, 3
    x1, x2, Hm = _pairs(B, h, w, seed=50)
    x1, x2, Hm = x1.to(dev), x2.to(dev), Hm.to(dev)
    with torch.no_grad():
        items = codec.compress_batch(x1, x2, Hm)
        out = codec.decompress_batch([(it["header"], it["payload"]) for it in items], Hm)
        for b in range(B):
            sl = slice(b, b + 1)
            enc = codec.compress(x1[sl], x2[sl], Hm[sl], f"p{b}", str(tmp_path))
            assert items[b]["header"] == (tmp_path / f"p{b}.npz").read_bytes()
            assert items[b]["payload"] == (tmp_path / f"p{b}.bin").read_bytes()
            assert items[b]["bpp_real"] == enc["bpp_real"]
            assert np.frombuffer(items[b]["header"][:4], np.uint16).tolist() == [h, w]
            dec = codec.decompress(None, None, Hm[sl], f"p{b}", str(tmp_path), device=dev)
            for k in dec:
                if k != "dectime":
                    assert torch.equal(out[k][sl], dec[k]), (b, k)
    pad = padding_for(h, w)
    want = _defined(codec, x1, x2, Hm, pad)
    for k in VIEWS:
        assert torch.equal(out[k], want[k])
    with pytest.raises(ValueError):                         # pairs of different original sizes still refused
        x = torch.zeros(1, 3, 201, 333, device=dev)
        other = codec.compress_batch(x, x, Hm[:1])[0]
        codec.decompress_batch([(items[0]["header"], items[0]["payload"]), (other["header"], other["payload"])],
                               Hm[:2])
