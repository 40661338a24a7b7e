"""g_s_conv4 in col2im form (csrc/deconv_img.cu): ConvTranspose2d(128, 3, k=5, s=2, p=2, op=1) [+ after_gdn] against
torch on the same 16-bit-rounded operands — odd strip counts, several CTA ranges per strip, batch, both formats."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("n,h,w", [(1, 8, 14), (1, 16, 20), (2, 32, 45), (1, 64, 136), (1, 304, 544)])
@pytest.mark.parametrize("igdn", [False, True])
def test_deconv_img_matches_torch(n, h, w, dt, igdn):
    from masic_b200.convplan import DeconvImgPlan
    from oracle import hsic as OH
    dev = torch.device("cuda:0")
    torch.manual_seed(h * 131 + w)
    x = torch.randn(n, h, w, 128, device=dev).to(dt)
    wt = torch.randn(128, 3, 5, 5, device=dev) / (128 * 6.25) ** 0.5
    b = torch.randn(3, device=dev) * 0.1
    out = torch.full((n, 3, 2 * h, 2 * w), 777.0, device=dev)
    beta = gamma = None
    if igdn:
        beta = OH.nonneg_init(torch.ones(3) + torch.rand(3)).to(dev)
        gamma = OH.nonneg_init(0.1 * torch.eye(3) + torch.rand(3, 3) * 0.02).to(dev)
    plan = DeconvImgPlan(x=x, weight=wt, bias=b, out=out, igdn_beta=beta, igdn_gamma=gamma)
    plan.launch()
    torch.cuda.synchronize()
    ref = F.conv_transpose2d(x.float().permute(0, 3, 1, 2), wt.to(dt).float(), b, stride=2, padding=2, output_padding=1)
    if igdn:
        ref = OH.gdn(ref.cpu(), beta.cpu(), gamma.cpu(), True).to(dev)
    assert bool(torch.isfinite(out).all())
    err = float((out - ref).abs().max())
    assert err <= 2e-4 * float(ref.abs().max()) + 1e-5, err
    plan.launch()                                    # a second launch writes the same image (ring state does not leak)
    torch.cuda.synchronize()
    assert float((out - ref).abs().max()) == err


@pytest.mark.parametrize("n,h,w", [(1, 16, 20), (2, 32, 48), (1, 152, 272)])
def test_after_conv_chain_on_tensor_cores_through_the_launchers(n, h, w):
    """The right view's decoder tail as the engine runs it: g_s_conv4 (col2im) + after_gdn writing 16-bit channels 0..2 of a
    channels-last image, the warp of x1_hat writing channels 4..6 (masic_warp_perspective_fwd), then after_conv
    (ConvTranspose2d(6, 3, 5, stride 1), MASIC.py:600,616) as a conv_tc plan over the pixel-folded view of that image with
    a planar (NCHW fp32) output — against torch on the same fp16-rounded inputs."""
    from masic_b200 import _lib, ops
    from masic_b200.convplan import ConvPlan, DeconvImgPlan, PackedConv, fold8_weights_5x5_s1
    from oracle import hsic as OH
    dev = torch.device("cuda:0")
    torch.manual_seed(7 * h + w)
    H, W = 2 * h, 2 * w
    XOFF, XPAD = _lib.IMG_XOFF, _lib.IMG_XPAD
    x = torch.randn(n, h, w, 128, device=dev).half()
    wt = torch.randn(128, 3, 5, 5, device=dev) / (128 * 6.25) ** 0.5
    b = torch.randn(3, device=dev) * 0.1
    beta = OH.nonneg_init(torch.ones(3) + torch.rand(3)).to(dev)
    gamma = OH.nonneg_init(0.1 * torch.eye(3) + torch.rand(3, 3) * 0.02).to(dev)
    ac_in = torch.zeros(n, H, W + XPAD, 8, dtype=torch.float16, device=dev)
    out32 = torch.empty(n, 3, H, W, device=dev)
    plan = DeconvImgPlan(x=x, weight=wt, bias=b, out=out32, igdn_beta=beta, igdn_gamma=gamma, out16=ac_in, out16_coff=0,
                         out16_xoff=XOFF)
    plan.launch()
    # the 16-bit copy is the fp32 image rounded once
    assert torch.equal(ac_in[:, :, XOFF:XOFF + W, :3].permute(0, 3, 1, 2), out32.half())
    only16 = torch.zeros_like(ac_in)
    DeconvImgPlan(x=x, weight=wt, bias=b, out=None, igdn_beta=beta, igdn_gamma=gamma, out16=only16, out16_coff=0,
                  out16_xoff=XOFF).launch()
    assert torch.equal(only16, ac_in)
    # warp: fp32 planes and the 16-bit copy at channels 3..5
    img = torch.rand(n, 3, H, W, device=dev)
    Hm = OH.synthetic_homography(n, seed=3).to(dev)
    T = ops.warp_prepare(Hm, (H, W), (H, W), False)
    w32 = torch.empty(n, 3, H, W, device=dev)
    ops.warp_perspective_into(img, T, (H, W), dst=w32, dst2=ac_in, dst2_coff=4)
    assert torch.equal(w32, ops.warp_perspective(img, Hm, (H, W)))
    assert torch.equal(ac_in[:, :, XOFF:XOFF + W, 4:7].permute(0, 3, 1, 2), w32.half())
    assert torch.equal(ac_in[:, :, XOFF:XOFF + W, :3].permute(0, 3, 1, 2), out32.half())     # channels 0..2 untouched
    assert float(ac_in[:, :, :XOFF].abs().max()) == 0 and float(ac_in[:, :, XOFF + W:].abs().max()) == 0
    assert float(ac_in[..., 3].abs().max()) == 0 and float(ac_in[..., 7].abs().max()) == 0
    # after_conv
    post = torch.nn.ConvTranspose2d(6, 3, 5, 1, 2).to(dev)
    wf, bf, tmask = fold8_weights_5x5_s1(post.weight, post.bias, transposed=True, slots=(0, 1, 2, 4, 5, 6))
    pk = PackedConv(ksize=5, c_in=64, c_out=48, n_tile=48, weight=wf, bias=bf, f16=_lib.FMT_F16)
    x2_hat = torch.full((n, 3, H, W), 777.0, device=dev)
    cp = ConvPlan(packed=pk, x=ac_in.view(n, H, (W + XPAD) // 8, 64), stride=1, tap_mask=tmask, w_in=W // 8,
                  out=x2_hat.view(n * 3, H, W // 8, 8), out_blk_images=True)
    cp.launch()
    torch.cuda.synchronize()
    with torch.no_grad():
        ref = F.conv_transpose2d(torch.cat((out32.half().float(), w32.half().float()), 1), post.weight.half().float(),
                                 post.bias, stride=1, padding=2)
    assert bool(torch.isfinite(x2_hat).all())
    assert float((x2_hat - ref).abs().max()) <= 1e-5 + 1e-5 * float(ref.abs().max())
