"""Full MASIC in the pair stream (test3_real.py): PairStream.attach_enhancement + submit(..., enhance=True) replays the
cross quality enhancement network right after the codec, reading the codec's buffers in place, and reports bpp, PSNR,
MS-SSIM and LPIPS of the enhanced pair.

Everything here is checked bit for bit against what a user gets today one call at a time: HSIC.forward, then
Independent_EN.forward on its outputs, then ops.ms_ssim / LPIPS on the result.  The enhanced MSE is also checked
against a float64 evaluation, with the tolerance of the codec-only criterion test (test_hsic_gpu.py)."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

BASE = {"bpp_y1", "bpp_y2", "bpp_z1", "bpp_z2", "mse1", "mse2", "loss"}
CODEC = {"codec_psnr1", "codec_psnr2", "codec_mse1", "codec_mse2"}
MS = {"msssim1", "msssim2", "msssim1_db", "msssim2_db"}
LP = {"lpips1", "lpips2"}
VIEWS = ("x1_hat", "x2_hat")


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from masic_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


def _codec(dev):
    from masic_b200.hsic import HSIC
    torch.manual_seed(0)
    return HSIC().eval().to(dev)


def _enhancer(dev, seed=3):
    """Seeded Independent_EN with its output conv scaled down: a small correction on top of the decode, the regime the
    trained network works in (test_cqe_gpu.py::test_cqe_psnr_regime)."""
    from masic_b200.cqe import Independent_EN
    torch.manual_seed(seed)
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


def _pairs(n, h, w, seed, u8=False):
    from oracle import hsic as OH
    g = torch.Generator().manual_seed(seed)
    if u8:
        x1 = torch.randint(0, 256, (n, 3, h, w), generator=g, dtype=torch.uint8)
        x2 = torch.randint(0, 256, (n, 3, h, w), generator=g, dtype=torch.uint8)
    else:
        x1, x2 = torch.rand(n, 3, h, w, generator=g), torch.rand(n, 3, h, w, generator=g)
    return x1, x2, OH.synthetic_homography(n, seed=seed + 1)


def _unit(x, dev):
    """What the stream feeds the codec: ToTensor's img.float().div(255) for 8-bit images."""
    x = x.to(dev)
    return x.float().div(255) if x.dtype == torch.uint8 else x


def _today(codec, en, x1, x2, Hm):
    """Today's test3 path for one pair: HSIC.forward, then Independent_EN.forward on its reconstructions."""
    with torch.no_grad():
        out = codec(x1, x2, Hm)
        return out, en(out["x1_hat"], out["x2_hat"], Hm)


def _masic_error():
    from masic_b200._lib import MasicError
    return MasicError


@pytest.mark.parametrize("u8", [False, True], ids=["float32", "uint8"])
@pytest.mark.parametrize("depth", [2, 3])
def test_enhanced_pair_is_bit_identical_to_forward(dev, depth, u8):
    """Pipelined submissions (results read one pair behind, so the slots rotate with pairs in flight): the enhanced pair
    read back by want_recon and exposed by enhanced_outputs() equals Independent_EN.forward on the codec's output."""
    codec, en = _codec(dev), _enhancer(dev)
    h, w, n = 192, 256, 5
    x1, x2, Hm = _pairs(n, h, w, seed=11, u8=u8)
    want = [_today(codec, en, _unit(x1[i:i + 1], dev), _unit(x2[i:i + 1], dev), Hm[i:i + 1].to(dev))[1]
            for i in range(n)]
    x1p, x2p, Hp = x1.pin_memory(), x2.pin_memory(), Hm.pin_memory()
    ps = codec.pair_stream(h, w, dev, depth=depth, lmbda=0.001)
    ps.attach_enhancement(en)
    tickets = []
    for i in range(n):
        tickets.append(ps.submit(x1p[i:i + 1], x2p[i:i + 1], Hp[i:i + 1], want_recon=True, enhance=True))
        if i >= 1:
            ps.result(tickets[i - 1])
            rec = ps.reconstructions(tickets[i - 1])
            for v, k in enumerate(VIEWS):
                assert torch.equal(rec[v], want[i - 1][k].cpu()), (i - 1, k)
    ps.result(tickets[-1])
    rec = ps.reconstructions(tickets[-1])
    enh = ps.enhanced_outputs()
    for v, k in enumerate(VIEWS):
        assert torch.equal(rec[v], want[-1][k].cpu())
        assert torch.equal(enh[k], want[-1][k])
    # and against the stream's own codec outputs, as a user of outputs() would call it
    o, hd = ps.outputs(), Hm[n - 1:n].to(dev)
    with torch.no_grad():
        direct = en(o["x1_hat"], o["x2_hat"], hd)
    for k in VIEWS:
        assert torch.equal(enh[k], direct[k])


def test_enhanced_criterion(dev):
    """bpp is the codec's; codec_psnr* / codec_mse* equal an enhance=False submission of the same pair exactly; the
    enhanced MSE matches float64 torch on the enhanced outputs; the loss uses the enhanced MSE."""
    codec, en = _codec(dev), _enhancer(dev)
    h, w, lmbda = 192, 256, 0.001
    x1, x2, Hm = _pairs(3, h, w, seed=21)
    x1p, x2p, Hp = x1.pin_memory(), x2.pin_memory(), Hm.pin_memory()
    ps = codec.pair_stream(h, w, dev, depth=2, lmbda=lmbda)
    ps.attach_enhancement(en)
    for i in range(3):
        r0 = ps.result(ps.submit(x1p[i:i + 1], x2p[i:i + 1], Hp[i:i + 1]))
        r1 = ps.result(ps.submit(x1p[i:i + 1], x2p[i:i + 1], Hp[i:i + 1], enhance=True))
        assert set(r0[3]) == BASE and set(r1[3]) == BASE | CODEC
        d0, d1 = r0[3], r1[3]
        assert r1[0] == r0[0] and all(d1[k] == d0[k] for k in ("bpp_y1", "bpp_y2", "bpp_z1", "bpp_z2"))
        assert (d1["codec_psnr1"], d1["codec_psnr2"]) == r0[1:3]
        assert (d1["codec_mse1"], d1["codec_mse2"]) == (d0["mse1"], d0["mse2"])
        enh = ps.enhanced_outputs()
        for v, (k, x) in enumerate(((VIEWS[0], x1), (VIEWS[1], x2))):
            mse = float(((enh[k].double() - x[i:i + 1].to(dev).double()) ** 2).mean())
            assert d1[f"mse{v + 1}"] == pytest.approx(mse, rel=2e-6)
            assert r1[1 + v] == pytest.approx(10 * math.log10(1 / mse), abs=1e-4)
            assert r1[1 + v] != d1[f"codec_psnr{v + 1}"]         # the enhancement changed the pair
        assert d1["loss"] == pytest.approx(lmbda * 255 ** 2 * (d1["mse1"] + d1["mse2"]) + r1[0], rel=1e-6)


@pytest.mark.parametrize("lpips_first", [True, False], ids=["lpips_then_enhancement", "enhancement_then_lpips"])
def test_enhanced_ms_ssim_and_lpips(dev, lpips_first):
    """msssim=True / lpips=True with enhance=True measure the enhanced pair, bit for bit what ops.ssim_per_channel and
    LPIPS give on enhanced_outputs(), for both normalize settings and either attach order; enhance=False submissions on
    the same stream keep measuring the codec's pair."""
    from masic_b200 import ops
    codec, en, lp = _codec(dev), _enhancer(dev), _lpips(dev)
    h, w = 192, 256
    x1, x2, Hm = _pairs(2, h, w, seed=31)
    x1p, x2p, Hp = x1.pin_memory(), x2.pin_memory(), Hm.pin_memory()
    ps = codec.pair_stream(h, w, dev, depth=2, lmbda=0.001)
    for normalize in (True, False):
        if lpips_first:
            ps.attach_lpips(lp, normalize=normalize)
            ps.attach_enhancement(en)
        else:
            ps.attach_enhancement(en)
            ps.attach_lpips(lp, normalize=normalize)
        for i in range(2):
            xs = (x1[i:i + 1].to(dev), x2[i:i + 1].to(dev))
            for enhance in (False, True):
                t = ps.submit(x1p[i:i + 1], x2p[i:i + 1], Hp[i:i + 1], msssim=True, lpips=True, enhance=enhance)
                r = ps.result(t)
                assert set(r[3]) == BASE | MS | LP | (CODEC if enhance else set())
                imgs = ps.enhanced_outputs() if enhance else ps.outputs()
                per_ch = ps.slots[t % ps.depth]["res_h"][8:14]
                for v, k in enumerate(VIEWS):
                    op = ops.ssim_per_channel(imgs[k], xs[v], 1.0, ops.MS_SSIM_WEIGHTS)
                    assert torch.equal(op.cpu().reshape(3), per_ch[3 * v:3 * v + 3])
                    assert r[3][f"msssim{v + 1}"] == pytest.approx(float(ops.ms_ssim(imgs[k], xs[v], data_range=1.0)),
                                                                   abs=1e-7)
                    assert r[3][f"lpips{v + 1}"] == float(lp(imgs[k], xs[v], normalize=normalize))


def test_default_path_is_untouched(dev):
    """enhance=False submissions interleaved with enhance=True ones return the same numbers, keys and outputs() as on a
    stream with nothing attached."""
    codec, en, lp = _codec(dev), _enhancer(dev), _lpips(dev)
    h, w = 192, 256
    x1, x2, Hm = _pairs(3, h, w, seed=41)
    x1p, x2p, Hp = x1.pin_memory(), x2.pin_memory(), Hm.pin_memory()
    plain = codec.pair_stream(h, w, dev, depth=2, lmbda=0.001)
    ps = codec.pair_stream(h, w, dev, depth=2, lmbda=0.001)
    ps.attach_enhancement(en)
    ps.attach_lpips(lp)
    for i in range(3):
        for msssim in (False, True):
            args = (x1p[i:i + 1], x2p[i:i + 1], Hp[i:i + 1])
            want = plain.result(plain.submit(*args, msssim=msssim))
            want_out = {k: v.clone() for k, v in plain.outputs().items()}
            ps.result(ps.submit(*args, msssim=True, lpips=True, enhance=True))
            got = ps.result(ps.submit(*args, msssim=msssim))
            assert got == want and set(got[3]) == set(want[3])
            assert set(ps.outputs()) == set(want_out)
            for k, v in ps.outputs().items():
                assert torch.equal(v, want_out[k]), k
            with pytest.raises(_masic_error()):
                ps.enhanced_outputs()                              # the last pair was not enhanced


def test_edges(dev):
    """enhance=True before attach raises; criterion=False with want_recon returns the enhanced pair; submit_patches
    forwards the flag; a re-attach after a weight change follows the new weights (and only then)."""
    from masic_b200.udh import Net
    from oracle import udh as OU
    codec, en = _codec(dev), _enhancer(dev)
    h, w = 192, 256
    x1, x2, Hm = _pairs(1, h, w, seed=51)
    x1p, x2p, Hp = x1.pin_memory(), x2.pin_memory(), Hm.pin_memory()
    xd1, xd2, Hd = x1.to(dev), x2.to(dev), Hm.to(dev)
    ps = codec.pair_stream(h, w, dev, depth=2, lmbda=0.001)
    with pytest.raises(_masic_error()):
        ps.submit(x1p, x2p, Hp, enhance=True)
    ps.attach_enhancement(en)

    _, want = _today(codec, en, xd1, xd2, Hd)
    t = ps.submit(x1p, x2p, Hp, criterion=False, want_recon=True, enhance=True)
    assert ps.result(t) is None
    rec = ps.reconstructions(t)
    for v, k in enumerate(VIEWS):
        assert torch.equal(rec[v], want[k].cpu())
        assert torch.equal(ps.enhanced_outputs()[k], want[k])

    torch.manual_seed(1)
    udh = Net().eval()
    with torch.no_grad():
        udh.fc[5].weight.mul_(200.0)                              # a homography far from identity (test_udh_gpu.py)
    ps.attach_homography_net(udh.to(dev))
    a, b, corners = OU.synthetic_patches(1, seed=2)
    rp = ps.result(ps.submit_patches(x1p, x2p, a.pin_memory(), b.pin_memory(), corners.pin_memory(), enhance=True,
                                     want_recon=True))
    h_udh = ps.eng.Hm.clone()
    enh_p = {k: v.clone() for k, v in ps.enhanced_outputs().items()}
    assert set(rp[3]) == BASE | CODEC
    rs = ps.result(ps.submit(x1p, x2p, h_udh.cpu().pin_memory(), enhance=True))
    assert rp == rs
    for k in VIEWS:
        assert torch.equal(ps.enhanced_outputs()[k], enh_p[k])

    with torch.no_grad():
        en.conv2.weight.mul_(2.0)
    _, want_new = _today(codec, en, xd1, xd2, Hd)
    assert not torch.equal(want_new["x1_hat"], want["x1_hat"])
    ps.result(ps.submit(x1p, x2p, Hp, enhance=True))
    for k in VIEWS:                                                # the attached engines hold a snapshot
        assert torch.equal(ps.enhanced_outputs()[k], want[k])
    ps.attach_enhancement(en)
    ps.result(ps.submit(x1p, x2p, Hp, enhance=True))
    for k in VIEWS:
        assert torch.equal(ps.enhanced_outputs()[k], want_new[k])


def test_bound_cqe_engine_reads_inputs_in_place(dev):
    """CQEEngine(inputs=...) keeps the caller's tensors as its inputs, equals the copying engine, refuses inputs of the
    wrong shape or dtype, and refuses run() arguments (it copies nothing)."""
    from masic_b200.cqe import CQEEngine
    en = _enhancer(dev)
    h, w = 64, 96
    x1, x2, Hm = _pairs(1, h, w, seed=61)
    xd1, xd2, Hd = x1.to(dev), x2.to(dev), Hm.to(dev).contiguous()
    sd = en.state_dict()
    eng = CQEEngine(sd, 1, h, w, dev, inputs=(xd1, xd2, Hd))
    assert eng.x1 is xd1 and eng.x2 is xd2 and eng.Hm is Hd
    out = eng.run()
    with torch.no_grad():
        want = en(xd1, xd2, Hd)
    for k in VIEWS:
        assert torch.equal(out[k], want[k])
    with pytest.raises(_masic_error()):
        eng.run(xd1, xd2, Hd)
    with pytest.raises(_masic_error()):
        CQEEngine(sd, 1, h, w, dev, inputs=(xd1, xd2, Hd.double()))
    with pytest.raises(_masic_error()):
        CQEEngine(sd, 1, h, w + 2, dev, inputs=(xd1, xd2, Hd))


def test_full_size_pair(dev):
    """1216x2176, depth 2: the enhanced pair equals Independent_EN.forward on the stream's codec outputs bit for bit."""
    codec, en = _codec(dev), _enhancer(dev)
    h, w = 1216, 2176
    x1, x2, Hm = _pairs(1, h, w, seed=71, u8=True)
    ps = codec.pair_stream(h, w, dev, depth=2)
    ps.attach_enhancement(en)
    r = ps.result(ps.submit(x1.pin_memory(), x2.pin_memory(), Hm.pin_memory(), enhance=True))
    o, enh = ps.outputs(), ps.enhanced_outputs()
    with torch.no_grad():
        want = en(o["x1_hat"], o["x2_hat"], Hm.to(dev))
    for k in VIEWS:
        assert torch.equal(enh[k], want[k])
    assert math.isfinite(r[1]) and math.isfinite(r[3]["codec_psnr1"])
