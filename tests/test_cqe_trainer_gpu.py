"""Training step of the cross quality enhancement network (CQETrainer) against torch autograd through
oracle/cqe.py in fp32 on the CPU, on the seeded weights and inputs of test_cqe_gpu.py's `_run`.

Loss: lmbda * 255^2 * (mse1 + mse2) of the enhanced pair against the originals.  Loss and both MSEs within 0.5 %.
Gradients: per parameter tensor, cosine and norm ratio against the oracle's, with the tolerances of TOL by module."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

# per parameter tensor: (cosine >=, |norm ratio - 1| <=), by module.  Measured on an NVIDIA B200 at the two sizes of
# test_cqe_train_gradients_match_oracle (profiles/r3_cqe_train_gradients.json):
#  * "conv": the 78 weights / biases of the Enhancement_Blocks and conv0 / conv1 / conv2 (bf16 activations and
#    gradients, fp32 accumulation through ~20 layers); measured cos >= 0.99998, norm within 0.4 %;
#  * "mask": mask2weights_unit, whose gradient reaches it through the softmax from per-pixel sums over the blends and
#    the fuse (whose scatter adds with fp32 atomics); measured cos >= 0.99995, norm within 1.4 %.
TOL = {"conv": (0.9999, 0.01), "mask": (0.9995, 0.03)}
LOSS_RTOL = 5e-3
LMBDA = 0.01


def _tol_class(name):
    return "mask" if name.startswith("mask2weights") else "conv"


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from masic_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


def _setup(h, w, batch, seed=200, gain=1.0, out_gain=1.0, noise=0.05):
    """test_cqe_gpu._run's seeded oracle and inputs; x*_hat = the originals plus noise (the codec's decode)."""
    from oracle.cqe import OracleIndependentEN
    from oracle.hsic import synthetic_homography
    torch.manual_seed(0)
    ora = OracleIndependentEN()
    with torch.no_grad():
        for n_, p_ in ora.named_parameters():
            if n_.endswith("weight") and p_.dim() == 4 and not n_.startswith("mask2weights"):
                p_.mul_(gain)
        ora.conv2.weight.mul_(out_gain)
        ora.conv2.bias.mul_(out_gain)
    g = torch.Generator().manual_seed(seed)
    x1 = torch.rand(batch, 3, h, w, generator=g)
    x2 = torch.rand(batch, 3, h, w, generator=g)
    x1h = x1 + noise * torch.randn(x1.shape, generator=g)
    x2h = x2 + noise * torch.randn(x2.shape, generator=g)
    Hm = synthetic_homography(batch, seed=5)
    Hm[:, 0, 2] *= 0.25
    return ora, x1h, x2h, x1, x2, Hm


def _oracle_grads(ora, x1h, x2h, x1, x2, Hm):
    from oracle.cqe import OracleIndependentEN
    ora.zero_grad(set_to_none=True)
    with torch.enable_grad():
        out = OracleIndependentEN.forward.__wrapped__(ora, x1h, x2h, Hm)
        mse1 = torch.mean((out["x1_hat"] - x1) ** 2)
        mse2 = torch.mean((out["x2_hat"] - x2) ** 2)
        loss = LMBDA * 255.0 ** 2 * (mse1 + mse2)
        loss.backward()
    grads = {n: p.grad.detach().clone() for n, p in ora.named_parameters()}
    return grads, (float(loss.detach()), float(mse1.detach()), float(mse2.detach()))


def _net(ora, dev):
    from masic_b200.cqe import Independent_EN
    net = Independent_EN()
    net.load_state_dict(ora.state_dict())
    return net.to(dev).train()


def _margins(net, want):
    out = []
    for name, p in net.named_parameters():
        a, b = want[name].double(), p.grad.detach().double().cpu()
        na, nb = float(a.norm()), float(b.norm())
        out.append((name, float((a * b).sum()) / (na * nb + 1e-300), nb / (na + 1e-300)))
    return out


def _record(case, margins, res, want):
    """The measured margins as one JSON line on stdout (shown with `pytest -s`; profiles/r3_cqe_train_gradients.json)."""
    import json
    rec = {"case": case, "tensors": len(margins), "device": torch.cuda.get_device_name(0),
           "loss_cuda": res["loss"], "loss_oracle": want[0], "mse1_cuda": res["mse1"], "mse1_oracle": want[1],
           "mse2_cuda": res["mse2"], "mse2_oracle": want[2]}
    for cls in TOL:
        ms = [m for m in margins if _tol_class(m[0]) == cls]
        rec[cls] = {"tensors": len(ms), "cos_min": min(m[1] for m in ms),
                    "cos_median": sorted(m[1] for m in ms)[len(ms) // 2],
                    "norm_ratio_min": min(m[2] for m in ms), "norm_ratio_max": max(m[2] for m in ms),
                    "worst": [[n, round(c, 6), round(r, 5)] for n, c, r in sorted(ms, key=lambda t: t[1])[:5]]}
    print("cqe_train_gradients " + json.dumps(rec))


def _check(margins):
    bad = []
    for name, cos, ratio in margins:
        cos_min, rtol = TOL[_tol_class(name)]
        if cos < cos_min or abs(ratio - 1.0) > rtol:
            bad.append((name, round(cos, 6), round(ratio, 5)))
    assert not bad, bad


def _dev(dev, *ts):
    return [t.to(dev) for t in ts]


@pytest.mark.parametrize("h,w,batch", [(64, 128, 2), (128, 192, 1)])
def test_cqe_train_gradients_match_oracle(dev, h, w, batch):
    ora, x1h, x2h, x1, x2, Hm = _setup(h, w, batch)
    want, wl = _oracle_grads(ora, x1h, x2h, x1, x2, Hm)
    net = _net(ora, dev)
    tr = net.trainer(batch, h, w, dev, lmbda=LMBDA)
    res = tr.step_grads(*_dev(dev, x1h, x2h, Hm, x1, x2))
    assert res["loss"] == pytest.approx(wl[0], rel=LOSS_RTOL)
    assert res["mse1"] == pytest.approx(wl[1], rel=LOSS_RTOL)
    assert res["mse2"] == pytest.approx(wl[2], rel=LOSS_RTOL)
    margins = _margins(net, want)
    assert len(margins) == 86
    _record(f"{batch}x{h}x{w}", margins, res, wl)
    _check(margins)


def test_cqe_flat_gradient_layout(dev):
    ora, *_ = _setup(64, 64, 1)
    net = _net(ora, dev)
    tr = net.trainer(1, 64, 64, dev)
    off = 0
    for name, p in net.named_parameters():
        g = tr.grad(name)
        assert g.data_ptr() == tr.flat_grad.data_ptr() + 4 * off and g.shape == p.shape, name
        off += p.numel()
    assert off == tr.flat_grad.numel() == sum(p.numel() for p in net.parameters())


def test_cqe_train_eager_equals_graph_and_updated_weights(dev):
    """The first call is issued eagerly, the next ones replay the graph: same gradients up to the order of the fuse
    scatter's atomics.  After optimizer.step() the replay re-packs the updated weights: gradients match the oracle on the
    updated state_dict."""
    ora, x1h, x2h, x1, x2, Hm = _setup(64, 128, 2)
    net = _net(ora, dev)
    tr = net.trainer(2, 64, 128, dev, lmbda=LMBDA)
    args = _dev(dev, x1h, x2h, Hm, x1, x2)
    tr.step_grads(*args)
    eager = tr.flat_grad.clone()
    tr.step_grads(*args)
    assert tr.graph is not None
    graph = tr.flat_grad.clone()
    off = 0
    for name, p in net.named_parameters():
        a, b = eager[off:off + p.numel()].double(), graph[off:off + p.numel()].double()
        off += p.numel()
        cos = float((a * b).sum() / (a.norm() * b.norm() + 1e-300))
        assert cos > 0.99999 and abs(float(b.norm() / a.norm()) - 1) < 1e-3, (name, cos)
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    opt.step()
    res = tr.step_grads(*args)
    ora.load_state_dict({k: v.cpu() for k, v in net.state_dict().items()})
    want, wl = _oracle_grads(ora, x1h, x2h, x1, x2, Hm)
    assert res["loss"] == pytest.approx(wl[0], rel=LOSS_RTOL)
    _check(_margins(net, want))


def _psnr(a, b):
    return 10 * math.log10(1.0 / float(torch.mean((a.double() - b.double()) ** 2)))


def test_cqe_short_training_raises_psnr(dev):
    """test_cqe_psnr_regime's noisy decode of a clean pair: 30 Adam steps raise the PSNR against the clean images."""
    ora, x1h, x2h, x1, x2, Hm = _setup(128, 192, 1, seed=7, out_gain=0.03, noise=0.02)
    net = _net(ora, dev)
    tr = net.trainer(1, 128, 192, dev, lmbda=LMBDA)
    args = _dev(dev, x1h, x2h, Hm, x1, x2)
    opt = torch.optim.Adam(net.parameters(), lr=1e-4)

    def psnrs():
        net.eval()
        with torch.no_grad():
            o = net(args[0], args[1], args[2])
        net.train()
        return _psnr(o["x1_hat"].cpu(), x1), _psnr(o["x2_hat"].cpu(), x2)
    p0 = psnrs()
    losses = [tr.train_step(*args, opt)["loss"] for _ in range(30)]
    p1 = psnrs()
    print("cqe short run: psnr", p0, "->", p1, "loss", losses[0], "->", losses[-1])
    assert losses[-1] < losses[0]
    assert p1[0] > p0[0] and p1[1] > p0[1], (p0, p1)


# ------------------------------------------------------------------ kernels
def _warp_T(Hm, h, w, invert=0):
    from masic_b200 import _lib
    from masic_b200.train_ops import _s
    T = torch.empty(Hm.shape[0], 3, 3, dtype=torch.float64, device=Hm.device)
    _lib.check(_lib.load().masic_warp_prepare(Hm.data_ptr(), Hm.shape[0], h, w, h, w, invert, T.data_ptr(), _s()),
               "masic_warp_prepare")
    return T


def test_feature_fuse_bwd_matches_autograd(dev):
    from masic_b200 import train_ops as T
    from oracle.hsic import synthetic_homography, warp
    n, h, w, c = 2, 37, 53, 32
    g = torch.Generator().manual_seed(3)
    s_ = torch.randn(n, h, w, c, generator=g).bfloat16()
    o_ = torch.randn(n, h, w, c, generator=g).bfloat16()
    wt = torch.softmax(torch.randn(n, 2, h, w, generator=g), dim=1)
    gf = torch.randn(n, h, w, 2 * c, generator=g).bfloat16()
    Hm = synthetic_homography(n, seed=5)
    Hm[:, 0, 2] *= 0.25
    sf, of = s_.float().permute(0, 3, 1, 2).requires_grad_(), o_.float().permute(0, 3, 1, 2).requires_grad_()
    wr = wt.clone().requires_grad_()
    fused = torch.cat((sf * wr[:, 1:2], warp(of, Hm) * wr[:, 0:1]), dim=1)
    fused.backward(gf.float().permute(0, 3, 1, 2))
    Td = _warp_T(Hm.to(dev), h, w)
    d_self = torch.zeros(n, h, w, c, dtype=torch.bfloat16, device=dev)
    d_other = torch.zeros(n, h, w, c, device=dev)
    dwt = torch.zeros(n, h, w, 2, device=dev)
    T.cqe_feature_fuse_bwd(gf.to(dev), s_.to(dev), o_.to(dev), wt.to(dev), Td, d_self, d_other, dwt)
    torch.cuda.synchronize()
    want_self = sf.grad.permute(0, 2, 3, 1)
    assert torch.allclose(d_self.float().cpu(), want_self, rtol=8e-3, atol=1e-6)
    want_other = of.grad.permute(0, 2, 3, 1)
    assert torch.allclose(d_other.cpu(), want_other, rtol=1e-4, atol=1e-4)
    assert torch.allclose(dwt.cpu(), wr.grad.permute(0, 2, 3, 1), rtol=1e-3, atol=1e-3)


def test_blend_images_bwd_matches_autograd(dev):
    from masic_b200 import train_ops as T
    n, h, w = 2, 29, 45
    g = torch.Generator().manual_seed(4)
    a, b = torch.rand(n, 3, h, w, generator=g), torch.rand(n, 3, h, w, generator=g)
    wt = torch.softmax(torch.randn(n, 2, h, w, generator=g), dim=1).requires_grad_()
    gout = torch.randn(n, h, w, 16, generator=g)
    out = torch.cat((a * wt[:, 0:1], b * wt[:, 1:2]), dim=1)
    out.backward(gout[..., :6].permute(0, 3, 1, 2))
    base = torch.randn(n, h, w, 2, generator=g)
    dwt = base.clone().to(dev)
    T.cqe_blend_images_bwd(gout.to(dev), a.to(dev), b.to(dev), dwt)
    torch.cuda.synchronize()
    assert torch.allclose(dwt.cpu(), base + wt.grad.permute(0, 2, 3, 1), rtol=1e-5, atol=1e-5)


def test_conv_act_out_store(dev):
    """The pre-residual activation store equals an act-only plan of the same layer bit for bit, and the plan's own
    output is bit-identical with and without it."""
    from masic_b200.convplan import ACT_LEAKY, ConvPlan, PackedConv
    n, h, w, c = 2, 40, 72, 64
    g = torch.Generator().manual_seed(5)
    x = torch.randn(n, h, w, c, generator=g).bfloat16().to(dev)
    r0 = torch.randn(n, h, w, c, generator=g).bfloat16().to(dev)
    r1 = torch.randn(n, h, w, c, generator=g).bfloat16().to(dev)
    wgt = (0.05 * torch.randn(c, c, 3, 3, generator=g)).to(dev)
    bias = (0.1 * torch.randn(c, generator=g)).to(dev)
    pk = PackedConv(ksize=3, c_in=c, c_out=c, n_tile=c, weight=wgt, bias=bias)
    act, out_a, out_b = (torch.zeros(n, h, w, c, dtype=torch.bfloat16, device=dev) for _ in range(3))
    ao = torch.full((n, h, w, 2 * c), 7.0, dtype=torch.bfloat16, device=dev)
    ConvPlan(packed=pk, x=x, out=act, act=ACT_LEAKY).launch()
    ConvPlan(packed=pk, x=x, out=out_a, act=ACT_LEAKY, residual0=r0, residual1=r1).launch()
    ConvPlan(packed=pk, x=x, out=out_b, act=ACT_LEAKY, residual0=r0, residual1=r1, act_out=ao, act_out_coff=c).launch()
    torch.cuda.synchronize()
    assert torch.equal(out_a, out_b)
    assert torch.equal(ao[..., c:], act)
    assert bool((ao[..., :c] == 7.0).all())


def test_act_bwd_bias_out_matches_in_place(dev):
    from masic_b200 import train_ops as T
    from masic_b200.convplan import ACT_LEAKY
    g = torch.Generator().manual_seed(6)
    grad = torch.randn(3, 17, 23, 96, generator=g).bfloat16().to(dev)
    y = torch.randn(3, 17, 23, 64, generator=g).bfloat16().to(dev)
    orig, src = grad.clone(), grad.clone()
    dst = torch.zeros(3, 17, 23, 64, dtype=torch.bfloat16, device=dev)
    b_in, b_out = torch.zeros(64, device=dev), torch.zeros(64, device=dev)
    T.act_bwd_bias_out(src, 32, 64, y, 0, ACT_LEAKY, dst, 0, b_out)
    T.act_bwd_bias(grad, 32, 64, y, 0, ACT_LEAKY, b_in)
    torch.cuda.synchronize()
    assert torch.equal(src, orig) and torch.equal(dst, grad[..., 32:96])
    assert torch.allclose(b_in, b_out, rtol=1e-6, atol=1e-5)


# ------------------------------------------------------------------ data parallel
def _dp_worker(rank, world, port, tmp):
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world, device_id=dev)
    try:
        ora, x1h, x2h, x1, x2, Hm = _setup(64, 128, 2)
        net = _net(ora, dev)
        tr = net.trainer(1, 64, 128, dev, lmbda=LMBDA)
        sl = slice(rank, rank + 1)
        opt = torch.optim.SGD(net.parameters(), lr=1e-3)
        tr.train_step(*_dev(dev, x1h[sl], x2h[sl], Hm[sl], x1[sl], x2[sl]), opt)
        torch.save({k: v.cpu() for k, v in net.state_dict().items()}, f"{tmp}/rank{rank}.pt")
    finally:
        dist.destroy_process_group()


def test_cqe_train_step_two_ranks(dev, tmp_path):
    """train_step on the two halves of a batch on two GPUs: both ranks end with identical parameters, and the update
    matches a single-GPU step on the whole batch within the parity tolerance."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import socket
    import torch.multiprocessing as mp
    ora, x1h, x2h, x1, x2, Hm = _setup(64, 128, 2)
    before = {k: v.clone() for k, v in ora.state_dict().items()}
    net = _net(ora, dev)
    tr = net.trainer(2, 64, 128, dev, lmbda=LMBDA)
    tr.train_step(*_dev(dev, x1h, x2h, Hm, x1, x2), torch.optim.SGD(net.parameters(), lr=1e-3))
    single = {k: v.cpu() for k, v in net.state_dict().items()}
    with socket.socket() as so:
        so.bind(("127.0.0.1", 0))
        port = so.getsockname()[1]
    mp.spawn(_dp_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "rank0.pt"), torch.load(tmp_path / "rank1.pt")
    bad = []
    for k in before:
        assert torch.equal(r0[k], r1[k]), k
        a, b = (single[k] - before[k]).double(), (r0[k] - before[k]).double()
        cos = float((a * b).sum() / (a.norm() * b.norm() + 1e-300))
        cos_min, rtol = TOL[_tol_class(k)]
        if cos < cos_min or abs(float(b.norm() / a.norm()) - 1) > rtol:
            bad.append((k, cos))
    assert not bad, bad
