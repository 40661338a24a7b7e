"""GPU parity of the image-domain kernels (warp, masks, small convs, GDN, packs) against oracle/
and torch fp32 on the same inputs.  Warp is a tolerance item (kornia is un-vendored: the
restatement in oracle/shims is the specification) — WARP_ATOL on [0,1] images."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
WARP_ATOL = 1e-4


def _t(a):
    return torch.from_numpy(np.asarray(a))


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from masic_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


def test_warp_and_masks_match_fixture(dev, golden_dir):
    from masic_b200 import ops
    fx = np.load(golden_dir / "warp.npz")
    img, Hm = _t(fx["img"]).to(dev), _t(fx["H"]).to(dev)
    out, out_bf = ops.warp_perspective(img, Hm, (40, 56), bf16_pitch=16)
    assert (out.cpu() - _t(fx["warped"])).abs().max() <= WARP_ATOL
    assert (out_bf[..., :3].float().permute(0, 3, 1, 2).cpu() - _t(fx["warped"])).abs().max() <= 5e-3
    assert float(out_bf[..., 3:].abs().max()) == 0.0
    m_r = ops.warp_perspective(None, Hm, (40, 56), ones_shape=(2, 1, 40, 56))
    m_l = ops.warp_perspective(m_r, Hm, (40, 56), invert=True)
    assert (m_r.cpu() - _t(fx["mask_R"])).abs().max() <= WARP_ATOL
    assert (m_l.cpu() - _t(fx["mask_L"])).abs().max() <= WARP_ATOL


def _warp_exact_f64(img, Hm):
    """Ground truth: src = M^-1 dst in pixel space, bilinear, zeros outside — all in float64."""
    b, c, h, w = img.shape
    ys, xs = torch.meshgrid(torch.arange(h, dtype=torch.float64), torch.arange(w, dtype=torch.float64), indexing="ij")
    pts = torch.stack((xs, ys, torch.ones_like(xs)), -1).reshape(-1, 3)
    out = torch.zeros(b, c, h * w, dtype=torch.float64)
    for i in range(b):
        q = pts @ torch.inverse(Hm[i].double()).T
        sx, sy = q[:, 0] / q[:, 2], q[:, 1] / q[:, 2]
        x0, y0 = torch.floor(sx), torch.floor(sy)
        for dy in (0, 1):
            for dx in (0, 1):
                xi, yi = x0 + dx, y0 + dy
                wgt = (1 - (sx - xi).abs()) * (1 - (sy - yi).abs())
                ok = (xi >= 0) & (xi < w) & (yi >= 0) & (yi < h)
                v = img[i].double()[:, yi.clamp(0, h - 1).long(), xi.clamp(0, w - 1).long()]
                out[i] += v * (wgt * ok)
    return out.view(b, c, h, w)


@pytest.mark.parametrize("h,w", [(128, 192), (1216, 2176)])
def test_warp_against_oracle(dev, h, w):
    """The fp32 kornia chain (the oracle) carries rounding noise of its own that grows with the image
    size (~2e-4 at 2176 px); the kernel evaluates coordinates in fp64.  So: the kernel must match the
    float64 ground truth to blend rounding, and differ from the oracle by no more than the oracle
    itself differs from the ground truth (and by <= WARP_ATOL where the oracle is that accurate)."""
    from masic_b200 import ops
    from oracle import hsic as OH
    g = torch.Generator().manual_seed(2)
    img = torch.rand(1, 3, h, w, generator=g)
    img = F.avg_pool2d(img, 3, 1, 1)                      # mild low-pass so the warp is non-trivial but smooth
    Hm = OH.synthetic_homography(1, seed=1)
    ref = OH.warp(img, Hm)
    exact = _warp_exact_f64(img, Hm)
    out = ops.warp_perspective(img.to(dev), Hm.to(dev), (h, w)).cpu()
    e_oracle = float((ref.double() - exact).abs().max())
    e_cuda = float((out.double() - exact).abs().max())
    d = float((out - ref).abs().max())
    print(f"warp {h}x{w}: |oracle-exact|={e_oracle:.3g} |cuda-exact|={e_cuda:.3g} |cuda-oracle|={d:.3g}")
    assert e_cuda <= 5e-6
    assert d <= max(WARP_ATOL, 1.5 * e_oracle)
    assert d <= 1e-3
    # identity homography reproduces the image (to interpolation rounding)
    ident = ops.warp_perspective(img.to(dev), torch.eye(3, device=dev)[None], (h, w))
    assert (ident.cpu() - img).abs().max() <= 1e-5


def test_fast_warp_and_fused_mask_are_bit_identical_to_the_generic_kernel(dev):
    """warp_fast_kernel (the engine's configurations: 3 / 1 channels) must reproduce warp_kernel bit for bit — a 4-channel
    image takes the generic kernel, its first three planes are the 3-channel image — and masic_warp_perspective_fwd
    writes the warp of the all-ones image (x1_mask_R, MASIC.py:636-638) from the same launch, equal to the separate
    ones-warp; ragged widths (not a multiple of the 256 pixels a block covers), border pixels included."""
    from masic_b200 import ops
    from oracle import hsic as OH
    g = torch.Generator().manual_seed(11)
    for h, w in ((128, 192), (200, 328), (64, 1000)):
        img = torch.rand(2, 3, h, w, generator=g).to(dev)
        Hm = OH.synthetic_homography(2, seed=3).to(dev)
        img4 = torch.cat([img, img[:, :1]], dim=1).contiguous()
        fast = ops.warp_perspective(img, Hm, (h, w))
        generic = ops.warp_perspective(img4, Hm, (h, w))
        assert torch.equal(fast, generic[:, :3]), (h, w)
        ones_sep = ops.warp_perspective(None, Hm, (h, w), ones_shape=(2, 1, h, w))
        T = ops.warp_prepare(Hm, (h, w), (h, w), False)
        out = torch.empty_like(img)
        ones = torch.empty(2, 1, h, w, device=dev)
        ops.warp_perspective_into(img, T, (h, w), dst=out, ones=ones)
        assert torch.equal(out, fast) and torch.equal(ones, ones_sep), (h, w)
        # the generic kernel's form of the same call (4 channels): the mask comes from a second launch
        out4 = torch.empty_like(img4)
        ones4 = torch.empty(2, 1, h, w, device=dev)
        ops.warp_perspective_into(img4, T, (h, w), dst=out4, ones=ones4)
        assert torch.equal(out4, generic) and torch.equal(ones4, ones_sep), (h, w)


def test_small_convs_against_torch(dev):
    from masic_b200 import ops
    from masic_b200.ops import ACT_RELU, GDN_FWD
    from oracle import hsic as OH
    torch.manual_seed(4)
    a, b = torch.rand(2, 3, 40, 56), torch.rand(2, 3, 40, 56)
    pre = torch.nn.Conv2d(6, 3, 5, 1, 2)
    beta = OH.nonneg_init(torch.ones(3) + torch.rand(3))
    gamma = OH.nonneg_init(0.1 * torch.eye(3) + torch.rand(3, 3) * 0.02)
    with torch.no_grad():
        ref = OH.gdn(pre(torch.cat((a, b), 1)), beta, gamma, False)
    out_bf = torch.empty(2, 40, 56, 16, dtype=ops.ACT16, device=dev)      # the inference engines' 16-bit format (fp16)
    out = torch.empty(2, 3, 40, 56, device=dev)
    ops.conv_small(a.to(dev), b.to(dev), pre.weight.to(dev), pre.bias.to(dev), ksize=5, stride=1, gdn=GDN_FWD,
                   beta=beta.to(dev), gamma=gamma.to(dev), out=out, out_bf16=out_bf)
    assert (out.cpu() - ref).abs().max() <= 2e-5
    assert (out_bf[..., :3].float().permute(0, 3, 1, 2).cpu() - ref).abs().max() <= 1e-3
    # ConvTranspose2d(6, 3, 5, stride=1) == after_conv (MASIC.py:600)
    post = torch.nn.ConvTranspose2d(6, 3, 5, 1, 2)
    with torch.no_grad():
        ref2 = post(torch.cat((a, b), 1))
    out2 = ops.conv_small(a.to(dev), b.to(dev), post.weight.to(dev), post.bias.to(dev), ksize=5, stride=1,
                          transposed_s1=True)
    assert (out2.cpu() - ref2).abs().max() <= 2e-5
    # mask2weights layer: conv3 s2 + ReLU on an odd-sized map
    m = torch.rand(1, 1, 37, 51)
    c = torch.nn.Conv2d(1, 3, 3, 2, 1)
    with torch.no_grad():
        ref3 = F.relu(c(m))
    out3 = ops.conv_small(m.to(dev), None, c.weight.to(dev), c.bias.to(dev), ksize=3, stride=2, act=ACT_RELU)
    assert out3.shape == ref3.shape and (out3.cpu() - ref3).abs().max() <= 1e-5
    sm, sm_nhwc = ops.softmax_channels(out3, nhwc_out=True)
    assert torch.allclose(sm.cpu(), torch.softmax(ref3, 1), atol=1e-6)
    assert torch.equal(sm_nhwc.permute(0, 3, 1, 2), sm)


@pytest.mark.parametrize("h,w", [(64, 96), (37, 51), (200, 333), (1216, 2176)])
def test_mask2weights_fused_matches_the_layer_chain(dev, h, w):
    """masic_mask2weights (one launch) against torch and, bit for bit, against the chain of four small-conv launches +
    softmax it replaces (MASIC.py:472-506)."""
    from masic_b200 import ops
    from masic_b200.ops import ACT_RELU
    torch.manual_seed(11)
    n = 2 if h < 1000 else 1
    m = (torch.rand(n, 1, h, w) > 0.3).float() * torch.rand(n, 1, h, w)
    layers = [torch.nn.Conv2d(1, 3, 3, 2, 1), torch.nn.Conv2d(3, 6, 3, 2, 1), torch.nn.Conv2d(6, 6, 3, 2, 1),
              torch.nn.Conv2d(6, 3, 3, 2, 1)]
    with torch.no_grad():
        for l in layers:
            l.weight.mul_(3.0)
        t = m
        for i, l in enumerate(layers):
            t = l(t)
            if i < 3:
                t = F.relu(t)
        ref = torch.softmax(t, 1)
    ws, bs = [l.weight.to(dev) for l in layers], [l.bias.to(dev) for l in layers]
    got, got_nhwc = ops.mask2weights(m.to(dev), ws, bs, nhwc_out=True)
    assert got.shape == ref.shape
    assert (got.cpu() - ref).abs().max() <= 2e-6
    assert torch.equal(got_nhwc.permute(0, 3, 1, 2), got)
    t = m.to(dev)
    for i in range(4):
        t = ops.conv_small(t, None, ws[i], bs[i], ksize=3, stride=2, act=ACT_RELU if i < 3 else 0)
    chain = ops.softmax_channels(t)
    assert torch.equal(chain, got)


def test_standalone_gdn_matches_reference_fixture(dev, golden_dir):
    from masic_b200.layers import GDN
    fx = np.load(golden_dir / "gdn.npz")
    for tag, inv in (("gdn", False), ("igdn", True)):
        layer = GDN(12, inverse=inv).eval()
        with torch.no_grad():
            layer.beta.copy_(_t(fx[f"{tag}/beta"]))
            layer.gamma.copy_(_t(fx[f"{tag}/gamma"]))
        layer = layer.to(dev)
        with torch.no_grad():
            y = layer(_t(fx[f"{tag}/x"]).to(dev))
        assert torch.allclose(y.cpu(), _t(fx[f"{tag}/y"]), rtol=2e-5, atol=1e-6)


def test_layout_packs_round_trip(dev):
    from masic_b200 import ops
    x = torch.rand(2, 3, 17, 23, device=dev)
    p = ops.nchw_to_nhwc_bf16(x, 16)
    assert p.dtype == ops.ACT16 and torch.equal(p[..., :3].permute(0, 3, 1, 2).float(), x.to(ops.ACT16).float())
    assert float(p[..., 3:].abs().max()) == 0
    # width % 4 == 0, three channels: the four-pixels-per-thread variant, plain and hi|lo (MASIC_FMT_SPLIT) formats
    from masic_b200 import _lib
    x4 = torch.rand(2, 3, 18, 24, device=dev)
    p4 = ops.nchw_to_nhwc_bf16(x4, 8)
    assert torch.equal(p4[..., :3].permute(0, 3, 1, 2).float(), x4.to(ops.ACT16).float()) and float(p4[..., 3:].abs().max()) == 0
    sp = torch.full((2, 18, 24 + _lib.IMG_XPAD, 8), 7.0, dtype=ops.ACT16, device=dev)
    _lib.check(_lib.load().masic_nchw_to_nhwc_bf16(x4.data_ptr(), 2, 3, 18, 24, sp.data_ptr(), 8, 24 + _lib.IMG_XPAD, _lib.IMG_XOFF,
                                                   _lib.FMT_F16 | _lib.FMT_SPLIT, torch.cuda.current_stream().cuda_stream), "pack")
    body = sp[:, :, _lib.IMG_XOFF:_lib.IMG_XOFF + 24]
    hi, lo = body[..., :3].permute(0, 3, 1, 2).float(), body[..., 3:6].permute(0, 3, 1, 2).float()
    assert torch.equal(hi, x4.half().float()) and float((hi + lo - x4).abs().max()) <= 2e-7
    assert float(body[..., 6:].abs().max()) == 0 and float((sp[:, :, :_lib.IMG_XOFF] - 7).abs().max()) == 0
    y = torch.rand(2, 9, 11, 200, device=dev)
    assert torch.equal(ops.nhwc_to_nchw_f32(y, 192), y[..., :192].permute(0, 3, 1, 2))


def test_launchers_refuse_what_the_kernels_cannot_use_in_place(dev):
    """The in-place launchers raise MasicError before launching anything when handed a 16-bit image whose rows are
    neither w_out nor w_out + IMG_XPAD pixels, a non-contiguous or wrong-dtype destination, or a CPU tensor: the
    refused destination and the valid fp32 destination of the same call keep their contents."""
    from masic_b200 import _lib, ops
    from masic_b200._lib import MasicError
    n, h, w = 2, 16, 24
    x = torch.rand(n, 3, h, w, device=dev)
    T = ops.warp_prepare(torch.eye(3, device=dev).repeat(n, 1, 1), (h, w), (h, w))
    dst = torch.full((n, 3, h, w), 7.0, device=dev)
    f16 = dict(dtype=torch.float16, device=dev)
    bad16 = [torch.zeros(n, h, w + 1, 8, **f16),                                  # rows neither w nor w + IMG_XPAD
             torch.zeros(n, h, w + 2 * _lib.IMG_XPAD, 8, **f16),
             torch.zeros(n, h, 8, w, **f16).transpose(2, 3),                      # non-contiguous
             torch.zeros(n, h, w, 8, dtype=torch.float32, device=dev),            # not a 16-bit dtype
             torch.zeros(n, h, w, 8, dtype=torch.float16)]                        # CPU
    for bad in bad16:
        for call in (lambda: ops.warp_perspective_into(x, T, (h, w), dst=dst, dst16=bad),
                     lambda: ops.warp_perspective_into(x, T, (h, w), dst=dst, dst2=bad, dst2_coff=4),
                     lambda: ops.nchw_to_nhwc_into(x, bad)):
            with pytest.raises(MasicError):
                call()
    bad32 = [torch.zeros(n, 3, w, h, device=dev).transpose(2, 3),                 # non-contiguous
             torch.zeros(n, 3, h, w, dtype=torch.float64, device=dev),            # wrong dtype
             torch.zeros(n, 3, h, w)]                                             # CPU
    for bad in bad32:
        with pytest.raises(MasicError):
            ops.warp_perspective_into(x, T, (h, w), dst=bad)
        with pytest.raises(MasicError):
            ops.softmax_channels_into(x, bad)
    for call in (lambda: ops.warp_perspective_into(x.cpu(), T, (h, w), dst=dst),          # a CPU input
                 lambda: ops.warp_perspective_into(x, T.cpu(), (h, w), dst=dst),
                 lambda: ops.softmax_channels_into(x.cpu(), dst)):
        with pytest.raises(MasicError):
            call()
    torch.cuda.synchronize()
    assert bool((dst == 7.0).all())
    assert all(float(b.abs().max()) == 0 for b in bad16 + bad32)
