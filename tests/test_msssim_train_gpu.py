"""Training for MS-SSIM on the GPU: masic_ms_ssim_bwd against float64 autograd of oracle/msssim.py, its determinism,
batch invariance and `addend`, and HSICTrainer(metric="ms-ssim") against the oracle's training step with CompressAI's
MS-SSIM rate-distortion loss."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import msssim as OM  # noqa: E402


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from masic_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


def _pair(n, h, w, seed, dev):
    """A smooth texture (bilinear upsampling of random cells plus a sinusoid) and the same with Gaussian noise:
    PSNR 25 to 35 dB across the planes."""
    g = torch.Generator(device=dev).manual_seed(seed)
    cells = torch.rand(n, 3, h // 6 + 2, w // 6 + 2, generator=g, device=dev)
    x = torch.nn.functional.interpolate(cells, size=(h, w), mode="bilinear", align_corners=False)
    yy = torch.arange(h, device=dev).view(1, 1, h, 1)
    xx = torch.arange(w, device=dev).view(1, 1, 1, w)
    x = (0.8 * x + 0.2 * torch.sin(0.3 * yy + 0.17 * xx) * 0.5 + 0.1).clamp(0, 1)
    db = 25.0 + 10.0 * torch.rand(n, 3, 1, 1, generator=g, device=dev)
    x_hat = (x + 10 ** (-db / 20) * torch.randn(n, 3, h, w, generator=g, device=dev)).clamp(0, 1)
    return x_hat.contiguous(), x.contiguous()


def _fwd_bwd(x_hat, x, scale, addend=None):
    from masic_b200 import train_ops as T
    n, c, h, w = x_hat.shape
    scratch, work = T.ms_ssim_buffers(n, c, h, w, x_hat.device)
    out = torch.empty(n, c, device=x_hat.device)
    g = torch.empty_like(x_hat)
    T.ms_ssim_fwd(x_hat, x, scratch, out)
    T.ms_ssim_grad(x_hat, x, scratch, scale, g, addend, work=work)
    return out, g, scratch


def _reference(x_hat, x, scale):
    xr = x_hat.double().requires_grad_()
    OM.ms_ssim_per_channel(xr, x.double(), data_range=1.0).sum().mul(scale).backward()
    return xr.grad


@pytest.mark.parametrize("n,h,w", [(2, 512, 896), (1, 1216, 2176), (1, 321, 483), (1, 161, 177), (4, 192, 256)])
def test_gradient_matches_float64_autograd(dev, n, h, w):
    x_hat, x = _pair(n, h, w, 10 + h, dev)
    scale = -0.37
    out, g, _ = _fwd_bwd(x_hat, x, scale)
    ref = _reference(x_hat, x, scale)
    torch.cuda.synchronize()
    assert torch.isfinite(g).all()
    assert float(out.min()) > 0.5                      # no level clamps: every plane has a gradient
    for i in range(n):
        for c in range(3):
            got, want = g[i, c].double(), ref[i, c]
            rel = float((got - want).norm() / want.norm())
            mx = float((got - want).abs().max() / want.abs().max())
            assert rel <= 1e-3 and mx <= 1e-3, (i, c, rel, mx)


def test_addend_is_added_exactly(dev):
    x_hat, x = _pair(2, 321, 483, 5, dev)
    add = torch.randn_like(x_hat)
    _, g0, _ = _fwd_bwd(x_hat, x, 0.25)
    _, g1, _ = _fwd_bwd(x_hat, x, 0.25, addend=add)
    assert torch.equal(g1, g0 + add)
    # in place: addend and dx are one buffer
    from masic_b200 import train_ops as T
    scratch, work = T.ms_ssim_buffers(2, 3, 321, 483, dev)
    out = torch.empty(2, 3, device=dev)
    buf = add.clone()
    T.ms_ssim_fwd(x_hat, x, scratch, out)
    T.ms_ssim_grad(x_hat, x, scratch, 0.25, buf, buf, work=work)
    assert torch.equal(buf, g1)


def test_deterministic_and_forward_untouched(dev):
    from masic_b200 import train_ops as T
    x_hat, x = _pair(2, 512, 896, 7, dev)
    scratch, work = T.ms_ssim_buffers(2, 3, 512, 896, dev)
    out = torch.empty(2, 3, device=dev)
    T.ms_ssim_fwd(x_hat, x, scratch, out)
    out0, scratch0 = out.clone(), scratch.clone()
    g1, g2 = torch.empty_like(x_hat), torch.empty_like(x_hat)
    T.ms_ssim_grad(x_hat, x, scratch, 1.0, g1, work=work)
    T.ms_ssim_grad(x_hat, x, scratch, 1.0, g2, work=work)
    assert torch.equal(g1, g2)
    assert torch.equal(out, out0) and torch.equal(scratch, scratch0)
    from masic_b200 import ops
    assert torch.equal(ops.ssim_per_channel(x_hat, x, 1.0, ops.MS_SSIM_WEIGHTS), out0)


def test_batch_invariant(dev):
    x_hat, x = _pair(4, 200, 264, 9, dev)
    _, g, _ = _fwd_bwd(x_hat, x, 1.0)
    for i in range(4):
        _, gi, _ = _fwd_bwd(x_hat[i:i + 1].contiguous(), x[i:i + 1].contiguous(), 1.0)
        assert torch.equal(gi, g[i:i + 1])
    for i, c in ((0, 0), (3, 2)):
        _, gp, _ = _fwd_bwd(x_hat[i:i + 1, c:c + 1].contiguous(), x[i:i + 1, c:c + 1].contiguous(), 1.0)
        assert torch.equal(gp[0, 0], g[i, c])


def test_clamped_plane_has_zero_gradient(dev):
    x_hat, x = _pair(1, 192, 256, 11, dev)
    both = torch.cat([x_hat, 1.0 - x], dim=0).contiguous()        # second image: every level's cs is negative
    out, g, _ = _fwd_bwd(both, x.repeat(2, 1, 1, 1).contiguous(), 1.0)
    assert float(out[1].abs().max()) == 0.0
    assert torch.isfinite(g).all() and float(g[1].abs().max()) == 0.0
    _, g0, _ = _fwd_bwd(x_hat, x, 1.0)
    assert torch.equal(g[0:1], g0)


# ----------------------------------------------------------------------------------------------- the trainer
def _oracle_msssim_step(oracle, x1, x2, Hm, noise, lmbda):
    """oracle/train.py's step with CompressAI's RateDistortionLoss(metric="ms-ssim") on both views."""
    import math

    from oracle import train as OT
    oracle.train()
    for p in oracle.parameters():
        p.grad = None
    out = OT.forward_train(oracle, x1, x2, Hm, noise)
    n, _, h, w = x1.shape
    bpp = sum(torch.log(v).sum() / (-math.log(2) * n * h * w) for v in out["likelihoods"].values())
    ms1 = OM.ms_ssim(out["x1_hat"], x1, data_range=1.0)
    ms2 = OM.ms_ssim(out["x2_hat"], x2, data_range=1.0)
    loss = lmbda * ((1 - ms1) + (1 - ms2)) + bpp
    loss.backward()
    aux = OT.aux_loss(oracle)
    aux.backward()
    grads = {k: (p.grad.clone() if p.grad is not None else torch.zeros_like(p)) for k, p in oracle.named_parameters()}
    return loss.item(), bpp.item(), ms1.item(), ms2.item(), grads


@pytest.mark.parametrize("batch,h,w,scale", [(1, 192, 256, 1.0), (2, 192, 192, 8.0)])
def test_trainer_gradients_match_oracle(dev, batch, h, w, scale):
    from test_trainer_gpu import LOSS_RTOL, _setup
    oracle, net, x1, x2, Hm, noise = _setup(batch, h, w, scale, dev)
    lmbda = 8.0
    loss, bpp, ms1, ms2, grads = _oracle_msssim_step(oracle, x1, x2, Hm, noise, lmbda)
    tr = net.trainer(batch, h, w, dev, lmbda=lmbda, metric="ms-ssim")
    args = (x1.to(dev), x2.to(dev), Hm.to(dev))
    nz = {k: v.to(dev) for k, v in noise.items()}
    res = tr.step_grads(*args, noise=nz)
    print("cuda", res, "oracle", loss, bpp, ms1, ms2)
    assert set(res) == {"loss", "bpp", "mse", "aux", "msssim1", "msssim2"}
    assert res["loss"] == pytest.approx(loss, rel=LOSS_RTOL)
    assert res["bpp"] == pytest.approx(bpp, rel=LOSS_RTOL)
    assert res["msssim1"] == pytest.approx(ms1, rel=LOSS_RTOL)
    assert res["msssim2"] == pytest.approx(ms2, rel=LOSS_RTOL)
    got = {name: p.grad.detach().cpu().double().clone() for name, p in torch.nn.Module.named_parameters(net)}
    bad = _out_of_tolerance(got, grads)
    print("\n".join(str(b) for b in bad))
    g1 = tr.flat_grad.clone()
    res2 = tr.step_grads(*args, noise=nz)
    assert res2["loss"] == pytest.approx(res["loss"], rel=1e-6)
    assert float((tr.flat_grad - g1).norm() / g1.norm()) < 1e-3      # only atomics' summation order differs
    if bad:
        # The hyper-analysis weights get the rate term's gradient alone: the same forward gives them the same
        # gradient whatever the metric.  Where one misses its bar, the MSE step of the same case (with its own
        # oracle) must miss it as well, and the MS-SSIM step must give what the MSE step gives.
        from oracle import train as OT
        *_, grads_mse, _ = OT.train_step_grads(oracle, x1, x2, Hm, noise, lmbda)
        net.trainer(batch, h, w, dev, lmbda=lmbda).step_grads(*args, noise=nz)
        got_mse = {name: p.grad.detach().cpu().double() for name, p in torch.nn.Module.named_parameters(net)}
        bad_mse = {b[0] for b in _out_of_tolerance(got_mse, grads_mse)}
        print("out of tolerance with metric='mse' too:", sorted(bad_mse))
        for name, *_ in bad:
            assert name.startswith(("_h_a1.", "_h_a2.")) and name in bad_mse, name
            assert float((got[name] - got_mse[name]).norm() / got_mse[name].norm()) < 1e-3, name


def _out_of_tolerance(got, want):
    from test_trainer_gpu import TOL, _tol_class
    bad = []
    for name, w in want.items():
        w, g = w.double(), got[name]
        nw, ng = float(w.norm()), float(g.norm())
        if nw < 1e-12:
            assert ng < 1e-9, name
            continue
        cos = float((w * g).sum() / (nw * ng + 1e-300))
        cos_min, norm_rtol = TOL[_tol_class(name)]
        if cos < cos_min or abs(ng / nw - 1.0) > norm_rtol:
            bad.append((name, round(cos, 5), round(ng / nw, 4), nw))
    return bad


def test_mse_metric_issues_the_same_step(dev):
    from masic_b200.hsic import HSIC
    from masic_b200.trainer import HSICTrainer
    net = HSIC().to(dev).train()
    a = HSICTrainer(net, 1, 192, 256, dev)
    b = HSICTrainer(net, 1, 192, 256, dev, metric="mse")
    c = net.trainer(1, 192, 256, dev, metric="ms-ssim")
    for t in (b, c):
        assert [n for n, _ in t.fwd_ops] == [n for n, _ in a.fwd_ops]
        assert [n for n, _ in t.bwd_ops] == [n for n, _ in a.bwd_ops]
    x = torch.rand(1, 3, 192, 256, device=dev)
    Hm = torch.eye(3, device=dev)[None]
    ra, rb = a.step_grads(x, x, Hm), b.step_grads(x, x, Hm)
    assert list(ra) == list(rb) == ["loss", "bpp", "mse", "aux"]


def test_msssim_training_lowers_the_loss(dev):
    from masic_b200.hsic import HSIC
    torch.manual_seed(0)
    net = HSIC().to(dev).train()
    tr = net.trainer(2, 256, 256, dev, lmbda=8.0, metric="ms-ssim")
    opt = torch.optim.Adam(net.parameters(), lr=1e-4)
    aux = torch.optim.Adam(net.aux_parameters(), lr=1e-3)
    pairs = [_pair(2, 256, 256, 100 + i, dev) for i in range(4)]
    Hm = torch.eye(3, device=dev).repeat(2, 1, 1)
    losses = []
    for step in range(150):
        x1, x2 = pairs[step % 4]
        losses.append(tr.train_step(x2, x1, Hm, opt, aux, clip_max_norm=1.0)["loss"])
    first, last = sum(losses[:20]) / 20, sum(losses[-20:]) / 20
    print("mean loss of the first / last 20 steps", first, last)
    assert all(torch.isfinite(torch.tensor(losses)))
    assert last < first
